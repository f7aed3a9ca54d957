"""Neighbour aggregation that consumes the reconstructed rows (north star part (d)).

The reference's models call DGL 2.1.0 (un-vendored): dglnn.SAGEConv(in, out, 'mean') three
times (gnn_model.py:78-81, forward :206-217) and dglnn.GraphConv(norm='both',
allow_zero_in_degree=True) (gnn_model.py:287).  DGL is not part of this image, so the sparse part
is restated here over a minimal bipartite block:

    Block.indptr  int64 [num_dst + 1]   CSR by destination
    Block.indices int32 [num_edges]     source ids local to the block
    destination nodes are the first num_dst source nodes (h_dst = h[:num_dst], gnn_model.py:211)

and runs through ttg_spmm_csr_fwd / ttg_spmm_csr_bwd of the C ABI.  The dense parts (Linear,
bias) stay in torch: they are library GEMMs, not part of the path.
"""
import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import torch
from torch import nn

import _ttg


# backward passes that scatter to source rows: gather over the transposed block (Block.transposed) where that is
# kept, instead of atomics
GATHER_BACKWARD = True


@dataclass
class Block:
    indptr: torch.Tensor       # int64 [num_dst + 1]
    indices: torch.Tensor      # int32 [E]
    num_src: int
    num_dst: int

    def num_dst_nodes(self):
        return self.num_dst

    def num_src_nodes(self):
        return self.num_src

    def in_degrees(self):
        return (self.indptr[1:] - self.indptr[:-1])

    def out_degrees(self):
        return torch.bincount(self.indices.long(), minlength=self.num_src)

    def int(self):
        return self

    def to(self, device):
        return Block(self.indptr.to(device), self.indices.to(device), self.num_src, self.num_dst)

    def dst_of_edge(self):
        """int64 [E]: the destination of every edge of the destination-major lists (kept with the block)."""
        d = getattr(self, "_dst_of_edge", None)
        if d is None:
            d = torch.repeat_interleave(torch.arange(self.num_dst, device=self.indptr.device), self.in_degrees())
            object.__setattr__(self, "_dst_of_edge", d)
        return d

    def edge_ids(self):
        """int32 [E]: 0 .. E - 1 (the identity edge map, for segment sums with the aggregation kernel)."""
        e = getattr(self, "_edge_ids", None)
        if e is None:
            e = torch.arange(self.indices.numel(), dtype=torch.int32, device=self.indptr.device)
            object.__setattr__(self, "_edge_ids", e)
        return e

    def transposed(self):
        """The block in source-major order, computed once and kept: (indptr_t int64 [num_src + 1], dst_t int32 [E],
        eid_t int32 [E]) -- edge k of that order goes to destination dst_t[k] and is edge eid_t[k] of the
        destination-major lists.  Backward passes that scatter to source rows become gathers over it."""
        t = getattr(self, "_transposed", None)
        if t is None:
            src = self.indices.long()
            order = torch.argsort(src, stable=True)
            dst = self.dst_of_edge()
            counts = torch.bincount(src, minlength=self.num_src)
            indptr_t = torch.zeros(self.num_src + 1, dtype=torch.int64, device=src.device)
            indptr_t[1:] = torch.cumsum(counts, 0)
            t = (indptr_t, dst[order].to(torch.int32).contiguous(), order.to(torch.int32).contiguous())
            object.__setattr__(self, "_transposed", t)
        return t


def _gather_backward(block) -> bool:
    """Scatter-free backward (an SpMM over the transposed block) where the block is, or looks, static: a
    full-graph block (square) transposes once and keeps it; a sampled block is used once and the transposition
    (a sort of its edges) would cost more than the atomics it saves."""
    return GATHER_BACKWARD and (getattr(block, "_transposed", None) is not None or block.num_src == block.num_dst)


def _spmm_backward(block, dout, F, mean, edge_weight):
    """dx [num_src][F] of out = aggregate(block, x): as a gather over the transposed block or by atomics."""
    dev = dout.device
    if _gather_backward(block):
        indptr_t, dst_t, eid_t = block.transposed()
        w_t = None
        if mean:
            w_t = getattr(block, "_inv_deg_t", None)
            if w_t is None:
                inv = 1.0 / block.in_degrees().clamp(min=1).to(torch.float32)
                w_t = inv[dst_t.long()].contiguous()
                object.__setattr__(block, "_inv_deg_t", w_t)
        if edge_weight is not None:
            we = edge_weight[eid_t.long()]
            w_t = we if w_t is None else (w_t * we)
            w_t = w_t.contiguous()
        dx = torch.empty((block.num_src, F), dtype=torch.float32, device=dev)
        rc = _ttg.lib().ttg_spmm_csr_fwd(block.num_src, F, _ttg.ptr(indptr_t), _ttg.ptr(dst_t), _ttg.ptr(w_t), 0,
                                         _ttg.ptr(dout), _ttg.ptr(dx), _ttg.stream_of(dev))
        _ttg.check(rc, "spmm_csr_fwd (transposed)")
        return dx
    dx = torch.zeros((block.num_src, F), dtype=torch.float32, device=dev)
    rc = _ttg.lib().ttg_spmm_csr_bwd(block.num_dst, F, _ttg.ptr(block.indptr), _ttg.ptr(block.indices),
                                     _ttg.ptr(edge_weight), 1 if mean else 0, _ttg.ptr(dout), _ttg.ptr(dx),
                                     _ttg.stream_of(dev))
    _ttg.check(rc, "spmm_csr_bwd")
    return dx


class _SpMM(torch.autograd.Function):
    @staticmethod
    def forward(ctx, block, x, mean, edge_weight):
        indptr, indices, num_dst = block.indptr, block.indices, block.num_dst
        _ttg.require_cuda(indptr, "indptr", torch.int64)
        _ttg.require_cuda(indices, "indices", torch.int32)
        x = _ttg.require_cuda(x.contiguous(), "x", torch.float32)
        dev = x.device
        F = x.size(1)
        with _ttg.on_device(dev):
            out = torch.empty((num_dst, F), dtype=torch.float32, device=dev)
            rc = _ttg.lib().ttg_spmm_csr_fwd(num_dst, F, _ttg.ptr(indptr), _ttg.ptr(indices),
                                             _ttg.ptr(edge_weight), 1 if mean else 0, _ttg.ptr(x),
                                             _ttg.ptr(out), _ttg.stream_of(dev))
            _ttg.check(rc, "spmm_csr_fwd")
        ctx.save_for_backward(edge_weight)
        ctx.block = block
        ctx.cfg = (F, mean)
        return out

    @staticmethod
    def backward(ctx, dout):
        (edge_weight,) = ctx.saved_tensors
        F, mean = ctx.cfg
        with _ttg.on_device(dout.device):
            dx = _spmm_backward(ctx.block, dout.to(torch.float32).contiguous(), F, mean, edge_weight)
        return None, dx, None, None


class _SpMMWithSelf(torch.autograd.Function):
    """(aggregate(block, x), x[:num_dst]) as ONE autograd node.  A SAGE layer reads its input
    twice (gnn_model.py:211-214: h_dst = h[:num_dst] for fc_self, all of h for the neighbour mean);
    as two nodes autograd materialises the slice's gradient as a zero-filled [num_src, F] tensor,
    copies into it and adds it to the aggregation's gradient -- five passes over num_src * F floats
    (0.5 ms per step at products shape).  Here the slice's gradient is added in place to the first
    num_dst rows of the aggregation's gradient."""

    @staticmethod
    def forward(ctx, block, x, mean):
        indptr, indices, num_dst = block.indptr, block.indices, block.num_dst
        _ttg.require_cuda(indptr, "indptr", torch.int64)
        _ttg.require_cuda(indices, "indices", torch.int32)
        x = _ttg.require_cuda(x.contiguous(), "x", torch.float32)
        dev = x.device
        F = x.size(1)
        with _ttg.on_device(dev):
            out = torch.empty((num_dst, F), dtype=torch.float32, device=dev)
            rc = _ttg.lib().ttg_spmm_csr_fwd(num_dst, F, _ttg.ptr(indptr), _ttg.ptr(indices), None,
                                             1 if mean else 0, _ttg.ptr(x), _ttg.ptr(out),
                                             _ttg.stream_of(dev))
            _ttg.check(rc, "spmm_csr_fwd")
        ctx.block = block
        ctx.cfg = (num_dst, F, mean)
        return out, x[:num_dst].clone()

    @staticmethod
    def backward(ctx, dout, dself):
        num_dst, F, mean = ctx.cfg
        with _ttg.on_device(dout.device):
            dx = _spmm_backward(ctx.block, dout.to(torch.float32).contiguous(), F, mean, None)
            dx[:num_dst].add_(dself)
        return None, dx, None


def aggregate_with_self(block: Block, x: torch.Tensor, mean: bool) -> Tuple[torch.Tensor, torch.Tensor]:
    """(neighbour aggregate, the destination nodes' own rows): see _SpMMWithSelf."""
    return _SpMMWithSelf.apply(block, x, mean)


def aggregate(block: Block, x: torch.Tensor, mean: bool,
              edge_weight: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[v] = (1/deg(v) if mean) * sum_{u in N_in(v)} w_uv * x[u]; rows without in-edges are 0."""
    return _SpMM.apply(block, x, mean, edge_weight)


def mean_agg_plan(g) -> torch.Tensor:
    """The work-item plan of ttg_mean_agg for a whole graph (sampler.CSRGraph or anything with int64 `indptr`,
    int32 `indices`), built once and kept with the graph like Block.transposed(): every layer and width reuses
    it.  Rebuilt if indptr is replaced or modified in place."""
    key = (g.indptr.data_ptr(), g.indptr._version, g.indptr.numel(), g.indices.numel())
    kept = getattr(g, "_mean_agg_plan", None)
    if kept is not None and kept[0] == key:
        return kept[1]
    n, e = g.indptr.numel() - 1, g.indices.numel()
    _ttg.require_cuda(g.indptr, "indptr", torch.int64)
    _ttg.require_cuda(g.indices, "indices", torch.int32)
    dev = g.indptr.device
    lib = _ttg.lib()
    plan_bytes = lib.ttg_mean_agg_plan_bytes(n, e)
    ws_bytes = lib.ttg_mean_agg_workspace_bytes(n, e, 1)
    if plan_bytes == 0 or ws_bytes == 0:
        raise RuntimeError("mean_agg_plan: %d nodes / %d edges out of range" % (n, e))
    with _ttg.on_device(dev):
        plan = torch.empty(plan_bytes, dtype=torch.uint8, device=dev)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)     # the scan's scratch, for this call only
        rc = lib.ttg_mean_agg_plan(n, e, _ttg.ptr(g.indptr), _ttg.ptr(plan), plan_bytes, _ttg.ptr(ws), ws_bytes,
                                   _ttg.stream_of(dev))
        _ttg.check(rc, "mean_agg_plan")
    object.__setattr__(g, "_mean_agg_plan", (key, plan))
    return plan


def aggregate_full(g, x: torch.Tensor) -> torch.Tensor:
    """out[v] = mean of x over the in-neighbours of v, for EVERY node of the graph g (zero rows for nodes without
    in-edges); not differentiable.  For full-neighbour inference: rows are cut into work items of at most 256
    edges (ttg_mean_agg), so a node with 40 k in-edges does not hold one warp for the whole call as it would in
    aggregate()'s one-warp-per-destination kernel.  Deterministic: the same bits from every call."""
    x = _ttg.require_cuda(x.contiguous(), "x", torch.float32)
    n, e = g.indptr.numel() - 1, g.indices.numel()
    if x.dim() != 2 or x.size(0) != n:
        raise RuntimeError("aggregate_full: x must be [num_nodes=%d, F], got %s" % (n, tuple(x.shape)))
    F = x.size(1)
    dev = x.device
    if n == 0:
        return torch.empty((0, F), dtype=torch.float32, device=dev)
    lib = _ttg.lib()
    with _ttg.on_device(dev):
        plan = mean_agg_plan(g)
        ws_bytes = lib.ttg_mean_agg_workspace_bytes(n, e, F)
        if ws_bytes == 0:
            raise RuntimeError("aggregate_full: F=%d out of range" % F)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        out = torch.empty((n, F), dtype=torch.float32, device=dev)
        rc = lib.ttg_mean_agg(n, e, F, _ttg.ptr(g.indptr), _ttg.ptr(g.indices), _ttg.ptr(plan), plan.numel(),
                              _ttg.ptr(x), _ttg.ptr(out), _ttg.ptr(ws), ws_bytes, _ttg.stream_of(dev))
        _ttg.check(rc, "mean_agg")
    return out


def aggregate_sharded(g, bounds: Sequence[int], blocks: Sequence[int], F: int, out: torch.Tensor) -> torch.Tensor:
    """aggregate_full for the destination nodes of one shard, the source rows split over row blocks
    (ttg_mean_agg_sharded): g holds the shard's in-lists (int64 indptr [num_dst + 1], int32 indices with GLOBAL
    source ids); block r is the device address (an int) of the rows of nodes [bounds[r], bounds[r + 1]), [rows][F]
    fp32, as mapped on out's device -- a peer GPU's buffer or any allocation.  Writes out [num_dst, F] and returns
    it; bit-identical to aggregate_full over the concatenated blocks."""
    n, e = g.indptr.numel() - 1, g.indices.numel()
    _ttg.require_cuda(out, "out", torch.float32)
    if out.dim() != 2 or tuple(out.shape) != (n, F):
        raise RuntimeError("aggregate_sharded: out must be [num_dst=%d, F=%d], got %s" % (n, F, tuple(out.shape)))
    world = len(blocks)
    if len(bounds) != world + 1 or not 1 <= world <= _ttg.TTG_MAX_PEERS:
        raise RuntimeError("aggregate_sharded: %d blocks and %d bounds (need 1..%d blocks and one bound more)"
                           % (world, len(bounds), _ttg.TTG_MAX_PEERS))
    dev = out.device
    lib = _ttg.lib()
    ws_bytes = lib.ttg_mean_agg_workspace_bytes(n, e, F)
    if ws_bytes == 0:
        raise RuntimeError("aggregate_sharded: %d nodes / %d edges / F=%d out of range" % (n, e, F))
    with _ttg.on_device(dev):
        plan = mean_agg_plan(g)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        b = (C.c_int64 * (world + 1))(*[int(x) for x in bounds])
        x = (C.c_void_p * world)(*[int(p) for p in blocks])
        rc = lib.ttg_mean_agg_sharded(n, e, F, _ttg.ptr(g.indptr), _ttg.ptr(g.indices), _ttg.ptr(plan), plan.numel(),
                                      world, b, x, _ttg.ptr(out), _ttg.ptr(ws), ws.numel(), _ttg.stream_of(dev))
        _ttg.check(rc, "mean_agg_sharded")
    return out


class SAGEConv(nn.Module):
    """GraphSAGE layer with DGL 2.1 `SAGEConv(in, out, 'mean')` semantics:
    out = fc_self(h_dst) + fc_neigh(mean_{u in N(v)} h_src[u]) + bias, the neighbour Linear being
    applied BEFORE the aggregation iff in_feats > out_feats (so the last 256 -> 47 layer gathers
    47-wide rows and the first 100 -> 256 layer gathers the raw reconstructed rows)."""

    def __init__(self, in_feats: int, out_feats: int, aggregator_type: str = "mean",
                 bias: bool = True):
        super().__init__()
        if aggregator_type != "mean":
            raise NotImplementedError("only the 'mean' aggregator of the reference models")
        self.in_feats, self.out_feats = in_feats, out_feats
        self.fc_self = nn.Linear(in_feats, out_feats, bias=False)
        self.fc_neigh = nn.Linear(in_feats, out_feats, bias=False)
        self.bias = nn.Parameter(torch.zeros(out_feats)) if bias else None
        gain = nn.init.calculate_gain("relu")
        nn.init.xavier_uniform_(self.fc_self.weight, gain=gain)
        nn.init.xavier_uniform_(self.fc_neigh.weight, gain=gain)

    def forward(self, block: Block, feat: Tuple[torch.Tensor, torch.Tensor]) -> torch.Tensor:
        h_src, h_dst = feat if isinstance(feat, tuple) else (feat, None)
        # h_dst is the first num_dst rows of h_src (how the reference calls its layers,
        # gnn_model.py:211-214): both reads of h_src then go through one autograd node
        head = h_dst is None or (h_dst.data_ptr() == h_src.data_ptr() and h_dst.dim() == 2
                                 and h_dst.size(0) == block.num_dst and h_dst.size(1) == h_src.size(1)
                                 and h_dst.stride() == h_src.stride())
        if head and self.in_feats <= self.out_feats and h_src.requires_grad:
            agg, h_dst = aggregate_with_self(block, h_src, mean=True)
            h_neigh = self.fc_neigh(agg)
        else:
            if h_dst is None:
                h_dst = h_src[:block.num_dst]
            h_neigh = self._neighbours(lambda h: aggregate(block, h, mean=True), h_src)
        out = self.fc_self(h_dst) + h_neigh
        if self.bias is not None:
            out = out + self.bias
        return out

    def _neighbours(self, mean_of, h_src: torch.Tensor) -> torch.Tensor:
        """fc_neigh of the neighbour mean, `mean_of` being the aggregation: DGL applies the Linear first when
        that shrinks the rows to gather (in_feats > out_feats), after the aggregation otherwise."""
        if self.in_feats > self.out_feats:
            return mean_of(self.fc_neigh(h_src))
        return self.fc_neigh(mean_of(h_src))

    @torch.no_grad()
    def forward_full(self, g, h: torch.Tensor) -> torch.Tensor:
        """The layer on every node of a whole graph g (sampler.CSRGraph; h [num_nodes, in_feats]): layer-wise
        full-neighbour inference (gnn_model.py:220-253), the neighbour mean by aggregate_full."""
        out = self.fc_self(h)
        out += self._neighbours(lambda x: aggregate_full(g, x), h)
        if self.bias is not None:
            out += self.bias
        return out

    def forward_aggregated(self, h_dst: torch.Tensor, h_mean: torch.Tensor) -> torch.Tensor:
        """The same layer when the caller already holds the destination rows and the neighbour mean
        (sage.SAGE with fuse_input: the TT lookup sums the neighbours' rows per destination itself)."""
        if self.in_feats > self.out_feats:
            raise NotImplementedError("forward_aggregated: this layer applies fc_neigh before the aggregation")
        out = self.fc_self(h_dst) + self.fc_neigh(h_mean)
        if self.bias is not None:
            out = out + self.bias
        return out


class GraphConv(nn.Module):
    """GCN layer with DGL `GraphConv(norm='both', allow_zero_in_degree=True)` semantics:
    h = D_in^-1/2 * A * (D_out^-1/2 * x) with degrees clamped to >= 1, weight applied before the
    aggregation iff in_feats > out_feats."""

    def __init__(self, in_feats: int, out_feats: int, norm: str = "both", bias: bool = True):
        super().__init__()
        if norm != "both":
            raise NotImplementedError("only norm='both' of the reference GCN")
        self.in_feats, self.out_feats = in_feats, out_feats
        self.weight = nn.Parameter(torch.empty(in_feats, out_feats))
        nn.init.xavier_uniform_(self.weight)
        self.bias = nn.Parameter(torch.zeros(out_feats)) if bias else None

    def forward(self, block: Block, feat: torch.Tensor) -> torch.Tensor:
        out_deg = block.out_degrees().clamp(min=1).to(torch.float32)
        x = feat * out_deg.pow(-0.5).unsqueeze(1)
        if self.in_feats > self.out_feats:
            rst = aggregate(block, x @ self.weight, mean=False)
        else:
            rst = aggregate(block, x, mean=False) @ self.weight
        in_deg = block.in_degrees().clamp(min=1).to(torch.float32)
        rst = rst * in_deg.pow(-0.5).unsqueeze(1)
        if self.bias is not None:
            rst = rst + self.bias
        return rst


# --------------------------------------------------------------------------------------------
# GAT (reference: class GATConv / GAT, gnn_model.py:300-497)
# --------------------------------------------------------------------------------------------
class _EdgeSoftmax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, indptr, score, num_dst):
        score = _ttg.require_cuda(score.contiguous(), "score", torch.float32)
        dev, H = score.device, score.size(1)
        with _ttg.on_device(dev):
            a = torch.empty_like(score)
            rc = _ttg.lib().ttg_edge_softmax_csr_fwd(num_dst, H, _ttg.ptr(indptr), _ttg.ptr(score),
                                                     _ttg.ptr(a), _ttg.stream_of(dev))
            _ttg.check(rc, "edge_softmax_csr_fwd")
        ctx.save_for_backward(indptr, a)
        ctx.num_dst = num_dst
        return a

    @staticmethod
    def backward(ctx, da):
        indptr, a = ctx.saved_tensors
        dev, H = a.device, a.size(1)
        with _ttg.on_device(dev):
            da = da.to(torch.float32).contiguous()
            ds = torch.empty_like(a)
            rc = _ttg.lib().ttg_edge_softmax_csr_bwd(ctx.num_dst, H, _ttg.ptr(indptr), _ttg.ptr(a),
                                                     _ttg.ptr(da), _ttg.ptr(ds), _ttg.stream_of(dev))
            _ttg.check(rc, "edge_softmax_csr_bwd")
        return None, ds, None


class _HeadSpMM(torch.autograd.Function):
    @staticmethod
    def forward(ctx, block, a, ft):
        indptr, indices, num_dst = block.indptr, block.indices, block.num_dst
        a = _ttg.require_cuda(a.contiguous(), "a", torch.float32)
        ft = _ttg.require_cuda(ft.contiguous(), "ft", torch.float32)      # [num_src][H][F]
        dev, H, F = ft.device, ft.size(1), ft.size(2)
        with _ttg.on_device(dev):
            out = torch.empty((num_dst, H, F), dtype=torch.float32, device=dev)
            rc = _ttg.lib().ttg_head_spmm_csr_fwd(num_dst, H, F, _ttg.ptr(indptr), _ttg.ptr(indices),
                                                  _ttg.ptr(a), _ttg.ptr(ft), _ttg.ptr(out),
                                                  _ttg.stream_of(dev))
            _ttg.check(rc, "head_spmm_csr_fwd")
        ctx.save_for_backward(indptr, indices, a, ft)
        ctx.num_dst = num_dst
        ctx.block = block
        return out

    @staticmethod
    def backward(ctx, dout):
        indptr, indices, a, ft = ctx.saved_tensors
        dev, H, F = ft.device, ft.size(1), ft.size(2)
        with _ttg.on_device(dev):
            dout = dout.to(torch.float32).contiguous()
            da = torch.empty_like(a)
            if _gather_backward(ctx.block):
                # dft by a gather over the transposed block (kept with the block: a static graph transposes once)
                # instead of 16-byte atomics into the source rows: 2x faster at ogbn-arxiv shape
                indptr_t, dst_t, eid_t = ctx.block.transposed()
                dft = torch.empty_like(ft)
                rc = _ttg.lib().ttg_head_spmm_csr_bwd_gather(
                    ctx.num_dst, ft.size(0), H, F, _ttg.ptr(indptr), _ttg.ptr(indices), _ttg.ptr(a), _ttg.ptr(ft),
                    _ttg.ptr(dout), _ttg.ptr(indptr_t), _ttg.ptr(dst_t), _ttg.ptr(eid_t), _ttg.ptr(dft),
                    _ttg.ptr(da), _ttg.stream_of(dev))
                _ttg.check(rc, "head_spmm_csr_bwd_gather")
            else:
                dft = torch.zeros_like(ft)
                rc = _ttg.lib().ttg_head_spmm_csr_bwd(ctx.num_dst, H, F, _ttg.ptr(indptr),
                                                      _ttg.ptr(indices), _ttg.ptr(a), _ttg.ptr(ft),
                                                      _ttg.ptr(dout), _ttg.ptr(dft), _ttg.ptr(da),
                                                      _ttg.stream_of(dev))
                _ttg.check(rc, "head_spmm_csr_bwd")
        return None, da, dft


class _EdgeAddUV(torch.autograd.Function):
    """score[e] = el[src(e)] + er[dst(e)] (DGL's u_add_v) on a block whose transposed form is kept: the backward
    sums d_score over each source's out-edges and each destination's in-edges with the aggregation kernel
    (rows of d_score gathered through the edge map / the identity) instead of torch's index_put with accumulate."""

    @staticmethod
    def forward(ctx, block, el, er):
        ctx.block = block
        return el[block.indices.long()] + er[block.dst_of_edge()]

    @staticmethod
    def backward(ctx, d):
        block = ctx.block
        d = _ttg.require_cuda(d.contiguous(), "d_score", torch.float32)
        H = d.size(1)
        dev = d.device
        indptr_t, _, eid_t = block.transposed()
        with _ttg.on_device(dev):
            d_el = torch.empty((block.num_src, H), dtype=torch.float32, device=dev)
            d_er = torch.empty((block.num_dst, H), dtype=torch.float32, device=dev)
            lib = _ttg.lib()
            _ttg.check(lib.ttg_spmm_csr_fwd(block.num_src, H, _ttg.ptr(indptr_t), _ttg.ptr(eid_t), None, 0,
                                            _ttg.ptr(d), _ttg.ptr(d_el), _ttg.stream_of(dev)), "u_add_v backward (src)")
            _ttg.check(lib.ttg_spmm_csr_fwd(block.num_dst, H, _ttg.ptr(block.indptr), _ttg.ptr(block.edge_ids()),
                                            None, 0, _ttg.ptr(d), _ttg.ptr(d_er), _ttg.stream_of(dev)),
                       "u_add_v backward (dst)")
        return None, d_el, d_er


def edge_add_uv(block: Block, el: torch.Tensor, er: torch.Tensor) -> torch.Tensor:
    """[E][H] scores el[src(e)] + er[dst(e)]."""
    if _gather_backward(block) and el.dtype == torch.float32 and er.dtype == torch.float32:
        return _EdgeAddUV.apply(block, el, er)
    return el[block.indices.long()] + er[block.dst_of_edge()]


def edge_softmax(block: Block, score: torch.Tensor) -> torch.Tensor:
    """softmax of score [E][H] over the in-edges of every destination node, per head."""
    return _EdgeSoftmax.apply(block.indptr, score, block.num_dst)


def attention_aggregate(block: Block, a: torch.Tensor, ft: torch.Tensor) -> torch.Tensor:
    """out[v, h, :] = sum_{e in N_in(v)} a[e, h] * ft[src(e), h, :]"""
    return _HeadSpMM.apply(block, a, ft)


class GATConv(nn.Module):
    """The reference's GATConv (gnn_model.py:318-440; same constructor keywords, parameter names
    and initialisation): attention scores by "first projection then addition", LeakyReLU, softmax
    over the in-edges, attention-weighted sum, optional symmetric degree normalisation
    (norm="both"), residual and activation.  Returns [num_dst, num_heads, out_feats]."""

    def __init__(self, in_feats, out_feats, num_heads=1, feat_drop=0.0, attn_drop=0.0,
                 negative_slope=0.2, residual=False, activation=None, allow_zero_in_degree=False,
                 norm="none"):
        super().__init__()
        if norm not in ("none", "both"):
            raise ValueError('Invalid norm value. Must be either "none", "both". But got "%s".' % norm)
        self._num_heads, self._out_feats, self._norm = num_heads, out_feats, norm
        self._in_src_feats, self._in_dst_feats = (in_feats if isinstance(in_feats, tuple)
                                                  else (in_feats, in_feats))
        self._allow_zero_in_degree = allow_zero_in_degree
        if isinstance(in_feats, tuple):
            self.fc_src = nn.Linear(self._in_src_feats, out_feats * num_heads, bias=False)
            self.fc_dst = nn.Linear(self._in_dst_feats, out_feats * num_heads, bias=False)
        else:
            self.fc = nn.Linear(self._in_src_feats, out_feats * num_heads, bias=False)
        self.attn_l = nn.Parameter(torch.empty(1, num_heads, out_feats))
        self.attn_r = nn.Parameter(torch.empty(1, num_heads, out_feats))
        self.feat_drop = nn.Dropout(feat_drop)
        self.attn_drop = nn.Dropout(attn_drop)
        self.leaky_relu = nn.LeakyReLU(negative_slope)
        if residual:
            self.res_fc = (nn.Linear(self._in_dst_feats, num_heads * out_feats, bias=False)
                           if self._in_dst_feats != out_feats else nn.Identity())
        else:
            self.register_buffer("res_fc", None)
        self._activation = activation
        self.reset_parameters()

    def reset_parameters(self):
        gain = nn.init.calculate_gain("relu")
        if hasattr(self, "fc"):
            nn.init.xavier_normal_(self.fc.weight, gain=gain)
        else:
            nn.init.xavier_normal_(self.fc_src.weight, gain=gain)
            nn.init.xavier_normal_(self.fc_dst.weight, gain=gain)
        nn.init.xavier_normal_(self.attn_l, gain=gain)
        nn.init.xavier_normal_(self.attn_r, gain=gain)
        if isinstance(self.res_fc, nn.Linear):
            nn.init.xavier_normal_(self.res_fc.weight, gain=gain)

    def set_allow_zero_in_degree(self, set_value):
        self._allow_zero_in_degree = set_value

    def forward(self, block: Block, feat):
        H, F = self._num_heads, self._out_feats
        if isinstance(feat, tuple):
            h_src, h_dst = self.feat_drop(feat[0]), self.feat_drop(feat[1])
            fc_src = self.fc_src if hasattr(self, "fc_src") else self.fc
            fc_dst = self.fc_dst if hasattr(self, "fc_dst") else self.fc
            feat_src = fc_src(h_src).view(-1, H, F)
            feat_dst = fc_dst(h_dst).view(-1, H, F)
        else:
            h_src = h_dst = self.feat_drop(feat)
            feat_src = self.fc(h_src).view(-1, H, F)
            feat_dst = feat_src[:block.num_dst]
            h_dst = h_dst[:block.num_dst]
        if self._norm == "both":
            degs = block.out_degrees().float().clamp(min=1)
            feat_src = feat_src * degs.pow(-0.5).view(-1, 1, 1)
        el = (feat_src * self.attn_l).sum(dim=-1)              # [num_src][H]
        er = (feat_dst * self.attn_r).sum(dim=-1)              # [num_dst][H]
        deg_in = block.in_degrees()
        e = self.leaky_relu(edge_add_uv(block, el, er))      # u_add_v
        a = self.attn_drop(edge_softmax(block, e))
        rst = attention_aggregate(block, a, feat_src)
        if self._norm == "both":
            rst = rst * deg_in.float().clamp(min=1).pow(0.5).view(-1, 1, 1)
        if self.res_fc is not None:
            rst = rst + self.res_fc(h_dst).view(h_dst.shape[0], -1, F)
        if self._activation is not None:
            rst = self._activation(rst)
        return rst


class _Bias(nn.Module):
    def __init__(self, size):
        super().__init__()
        self.bias = nn.Parameter(torch.zeros(size))

    def forward(self, x):
        return x + self.bias


class GAT(nn.Module):
    """The reference's GAT model (gnn_model.py:444-497): GATConv + a parallel Linear per layer,
    BatchNorm / activation / dropout between layers, mean over heads and a bias at the end."""

    def __init__(self, in_feats, n_classes, n_hidden, n_layers, n_heads, activation, dropout=0.0,
                 attn_drop=0.0, norm="none"):
        super().__init__()
        self.n_layers, self.num_heads = n_layers, n_heads
        self.convs, self.linear, self.bns = nn.ModuleList(), nn.ModuleList(), nn.ModuleList()
        for i in range(n_layers):
            in_hidden = n_heads * n_hidden if i > 0 else in_feats
            out_hidden = n_hidden if i < n_layers - 1 else n_classes
            self.convs.append(GATConv(in_hidden, out_hidden, num_heads=n_heads, attn_drop=attn_drop,
                                      norm=norm))
            self.linear.append(nn.Linear(in_hidden, n_heads * out_hidden, bias=False))
            if i < n_layers - 1:
                self.bns.append(nn.BatchNorm1d(n_heads * out_hidden))
        self.bias_last = _Bias(n_classes)
        self.dropout0 = nn.Dropout(min(0.1, dropout))
        self.dropout = nn.Dropout(dropout)
        self.activation = activation

    def forward(self, graph: Block, feat):
        h = self.dropout0(feat)
        for i in range(self.n_layers):
            conv = self.convs[i](graph, h)
            h = conv + self.linear[i](h[:graph.num_dst]).view(conv.shape)
            if i < self.n_layers - 1:
                h = self.dropout(self.activation(self.bns[i](h.flatten(1))))
        return self.bias_last(h.mean(1))


class GCN(nn.Module):
    """The reference's GCN model (gnn_model.py:269-314): GraphConv(norm='both') layers (bias only
    on the last), an optional parallel Linear per layer, BatchNorm / activation / dropout between
    layers.  `graph` is a Block with num_src == num_dst (the full graph, CSR by destination)."""

    def __init__(self, in_feats, n_hidden, n_classes, n_layers, activation, dropout, use_linear):
        super().__init__()
        self.n_layers, self.n_hidden, self.n_classes, self.use_linear = n_layers, n_hidden, n_classes, use_linear
        self.convs, self.bns = nn.ModuleList(), nn.ModuleList()
        if use_linear:
            self.linear = nn.ModuleList()
        for i in range(n_layers):
            in_hidden = n_hidden if i > 0 else in_feats
            out_hidden = n_hidden if i < n_layers - 1 else n_classes
            self.convs.append(GraphConv(in_hidden, out_hidden, "both", bias=(i == n_layers - 1)))
            if use_linear:
                self.linear.append(nn.Linear(in_hidden, out_hidden, bias=False))
            if i < n_layers - 1:
                self.bns.append(nn.BatchNorm1d(out_hidden))
        self.dropout0 = nn.Dropout(min(0.1, dropout))
        self.dropout = nn.Dropout(dropout)
        self.activation = activation

    def forward(self, graph: Block, feat):
        h = self.dropout0(feat)
        for i in range(self.n_layers):
            conv = self.convs[i](graph, h)
            h = conv + self.linear[i](h) if self.use_linear else conv
            if i < self.n_layers - 1:
                h = self.dropout(self.activation(self.bns[i](h)))
        return h
