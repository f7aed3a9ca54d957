"""GraphSAGE over TT-compressed node embeddings: the model of the reference's
sage_dgl_partition.py (class SAGE, gnn_model.py:44-217) on this package's operators --
TTEmbeddingBag for the input features, gnn_ops.SAGEConv for the layers, sampler.NeighborSampler
for the minibatches -- plus the synthetic ogbn-products-shaped graph the benchmarks run on
(there is no network for datasets; shapes from SURVEY 8d "G").
"""
from typing import List, Optional, Sequence

import torch
import torch.nn.functional as F
from torch import nn

import dp
from FBTT.tt_embeddings_ops import OptimType, TTEmbeddingBag
from gnn_ops import Block, SAGEConv, mean_agg_plan
from sampler import CSRGraph


class SAGE(nn.Module):
    """n_layers SAGEConv('mean') layers (in -> hidden -> ... -> classes, gnn_model.py:76-81) on
    top of a TTEmbeddingBag (gnn_model.py:113-125); forward as gnn_model.py:196-217."""

    def __init__(self, num_nodes: int, in_feats: int, n_hidden: int, n_classes: int,
                 n_layers: int = 3, dropout: float = 0.5, tt_rank: Sequence[int] = (16, 16),
                 p_shapes: Optional[Sequence[int]] = None, q_shapes: Optional[Sequence[int]] = None,
                 sparse: bool = True, learning_rate: float = 0.01, embed_name: str = "fbtt",
                 device=None, fuse_input: bool = False):
        """fuse_input (fbtt only): the first layer's neighbour mean comes out of the TT lookup itself -- one
        EmbeddingBag call whose bags are the destination nodes (one index each) followed by every destination's
        sampled neighbours (gnn_model.py:199-217 reconstructs all num_src rows and lets the layer gather them:
        [num_src, in_feats] written and read again every step).
        embed_name: "fbtt" (TTEmbeddingBag, --emb-name fbtt of the reference drivers) or "eff"
        (Eff_TTEmbedding, Efficient_TT/efficient_tt.py:214-307: forward by prefix reuse, backward = the
        fused SGD update of the cores, no gradient reaches autograd)."""
        super().__init__()
        self.embed_name = embed_name
        self.fuse_input = bool(fuse_input) and embed_name == "fbtt" and in_feats <= n_hidden
        self.layers = nn.ModuleList()
        self.layers.append(SAGEConv(in_feats, n_hidden, "mean"))
        for _ in range(1, n_layers - 1):
            self.layers.append(SAGEConv(n_hidden, n_hidden, "mean"))
        self.layers.append(SAGEConv(n_hidden, n_classes, "mean"))
        self.dropout = nn.Dropout(dropout)
        if embed_name == "eff":
            from Efficient_TT.efficient_tt import Eff_TTEmbedding
            dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
            self.embed_layer = Eff_TTEmbedding(
                num_embeddings=num_nodes, embedding_dim=in_feats, tt_ranks=list(tt_rank),
                tt_p_shapes=list(p_shapes) if p_shapes else None,
                tt_q_shapes=list(q_shapes) if q_shapes else None, learning_rate=learning_rate,
                weight_dist="uniform", device=dev.index or 0, batch_size=4096)
        elif embed_name == "fbtt":
            self.embed_layer = TTEmbeddingBag(
                num_embeddings=num_nodes, embedding_dim=in_feats, tt_ranks=list(tt_rank),
                tt_p_shapes=list(p_shapes) if p_shapes else None,
                tt_q_shapes=list(q_shapes) if q_shapes else None, sparse=sparse,
                optimizer=OptimType.SGD, learning_rate=learning_rate, use_cache=False,
                weight_dist="normal")
        else:
            raise ValueError("Unknown embedding type %r" % (embed_name,))   # gnn_model.py:126

    def dense_parameters(self) -> List[nn.Parameter]:
        return [p for layer in self.layers for p in layer.parameters()]

    def forward(self, blocks: Sequence[Block], input_nodes: torch.Tensor) -> torch.Tensor:
        first = 0
        if self.fuse_input:
            h = self._fused_first_layer(blocks[0], input_nodes)
            if len(self.layers) > 1:
                h = self.dropout(F.relu(h))
            first = 1
        elif self.embed_name == "eff":
            h = self.embed_layer(input_nodes)
        else:
            offsets = torch.arange(input_nodes.numel() + 1, device=input_nodes.device)
            h = self.embed_layer(input_nodes, offsets)
        for l in range(first, len(self.layers)):
            layer, block = self.layers[l], blocks[l]
            h = layer(block, (h, h[:block.num_dst]))
            if l != len(self.layers) - 1:
                h = self.dropout(F.relu(h))
        return h

    @torch.no_grad()
    def inference(self, g: CSRGraph) -> torch.Tensor:
        """[num_nodes, n_classes] logits of every node of g with ALL its in-neighbours, computed layer by layer
        over the whole graph (gnn_model.py:220-253): the rows of all nodes, then each layer on every node
        (SAGEConv.forward_full), ReLU between layers, no dropout.  The same for fuse_input on or off; the cores,
        the dense parameters and self.training are left as they are."""
        h = self._all_rows(g.num_nodes)
        for l, layer in enumerate(self.layers):
            h = layer.forward_full(g, h)
            if l != len(self.layers) - 1:
                h = F.relu_(h)
        return h

    def _all_rows(self, n: int) -> torch.Tensor:
        """Input features of nodes 0 .. n - 1: the row kernel on an implicit range where the table has one
        (ttg_tt_rows_range), else the lookup on arange(n) as the reference does (gnn_model.py:228-231)."""
        emb = self.embed_layer
        if n > emb.num_embeddings:
            raise RuntimeError("SAGE.inference: the graph has %d nodes, the embedding %d rows"
                               % (n, emb.num_embeddings))
        dev = emb.tt_cores[0].device
        ids = torch.arange(n, device=dev)
        if self.embed_name == "eff":
            return emb(ids)
        rows = emb.rows_range(0, n)
        if rows is not None:
            return rows
        return emb(ids, torch.arange(n + 1, device=dev))

    def _fused_first_layer(self, block: Block, input_nodes: torch.Tensor) -> torch.Tensor:
        """Bags 0 .. num_dst - 1: the destination nodes themselves; bags num_dst .. 2 num_dst - 1: their
        sampled neighbours, summed by the lookup (pooling "sum" of TTEmbeddingBag) and divided by the
        in-degree here.  One lookup, one backward, one fused update of the cores -- the same gradient as
        gathering reconstructed rows, since the mean is linear in them."""
        nd = block.num_dst
        dev = input_nodes.device
        idx = torch.cat([input_nodes[:nd], input_nodes[block.indices.long()]])
        offsets = torch.cat([torch.arange(nd, device=dev, dtype=torch.int64), block.indptr.to(torch.int64) + nd])
        out = self.embed_layer(idx, offsets)
        deg = block.in_degrees().clamp(min=1).to(torch.float32)
        h_mean = out[nd:] / deg.unsqueeze(1)
        return self.layers[0].forward_aggregated(out[:nd], h_mean)


@torch.no_grad()
def evaluate(model: SAGE, g: CSRGraph, labels: torch.Tensor, val_nid: torch.Tensor, test_nid: torch.Tensor):
    """(validation accuracy, test accuracy, logits of every node) of the full-neighbour inference, as the
    reference's evaluate (sage_dgl_partition.py:366-371): eval mode, SAGE.inference, accuracy of the argmax on
    each node set, train mode again."""
    model.eval()
    try:
        pred = model.inference(g)
    finally:
        model.train()
    hit = pred.argmax(1) == labels.to(pred.device)
    val_acc = float(hit[val_nid.to(pred.device)].float().mean())
    test_acc = float(hit[test_nid.to(pred.device)].float().mean())
    return val_acc, test_acc, pred


def shard_bounds(indptr: torch.Tensor, world: int) -> List[int]:
    """world + 1 node ids splitting nodes 0 .. N - 1 into contiguous shards of about equal weight, a node
    weighing deg(v) + ceil(E / N): bounds[r] is the first node whose prefix weight reaches r / world of the
    total (a search on indptr, so every rank derives the same bounds).  Shards may be empty when world > N."""
    n = indptr.numel() - 1
    e = int(indptr[-1]) if n > 0 else 0
    c = -(-e // max(n, 1))
    total = e + n * c
    prefix = indptr.to(torch.int64) + torch.arange(n + 1, dtype=torch.int64, device=indptr.device) * c
    targets = torch.tensor([r * total // world for r in range(1, world)], dtype=torch.int64, device=indptr.device)
    inner = torch.searchsorted(prefix, targets).tolist()
    return [0] + [min(int(b), n) for b in inner] + [n]


def check_bounds(bounds: Sequence[int], n: int, world: int) -> List[int]:
    """Caller shard bounds as ints: world + 1 non-decreasing node ids from 0 to n, else ValueError."""
    b = [int(x) for x in bounds]
    if len(b) != world + 1:
        raise ValueError("ShardedInference: %d bounds for %d ranks, need %d" % (len(b), world, world + 1))
    if b[0] != 0 or b[-1] != n:
        raise ValueError("ShardedInference: bounds must run from 0 to %d nodes, got %d .. %d" % (n, b[0], b[-1]))
    if any(b[r + 1] < b[r] for r in range(world)):
        raise ValueError("ShardedInference: bounds decrease: %s" % (b,))
    return b


class _DeviceRegion:
    """A [rows, F] fp32 window of a peer buffer as a torch tensor (torch.as_tensor reads the interface and
    shares the memory; the buffer outlives every view, see ShardedInference.close)."""

    def __init__(self, ptr: int, rows: int, F: int):
        self.__cuda_array_interface__ = {"shape": (rows, F), "typestr": "<f4", "data": (ptr, False),
                                         "strides": None, "version": 2}


class ShardedInference:
    """SAGE.inference sharded over the GPUs of one node, one process per GPU (collective calls).  Rank r owns
    nodes [bounds[r], bounds[r + 1]) and computes every layer for them only; the neighbour rows of other
    shards are read straight from the peers' memory over NVLink (gnn_ops.aggregate_sharded on buffers mapped
    by dp.map_peer_buffers), so no GPU holds a whole activation.

        inf = ShardedInference(model, g)      # bounds=None: contiguous shards balanced by deg(v) + ceil(E / N)
        logits = inf.inference()              # [hi - lo, n_classes]: model.inference(g)[lo:hi]
        val_acc, test_acc = inf.evaluate(labels, val_nid, test_nid)    # the same numbers on every rank
        inf.close()

    Every rank holds the same graph and the same model (checked: a checksum of the dense layers and the cores
    is compared across ranks, and every rank raises on a mismatch).  Caller bounds (e.g. the parts of
    reorder_graph(g, "kway", world)) are taken as given.  Each rank's peer buffer holds its rows of the layer
    input, the layer output and the projected input (fc_neigh first when a layer shrinks its rows), sized for
    the widest layer.  Writes and remote reads of a region are ordered by a stream-ordered barrier (an
    all-reduce of one element on the current stream), with no host synchronisation per layer.  The cores,
    the parameters and model.training are left as they are."""

    _IN, _OUT, _PROJ = 0, 1, 2

    def __init__(self, model: SAGE, g: CSRGraph, group=None, bounds: Optional[Sequence[int]] = None):
        import torch.distributed as dist
        from gnn_ops import aggregate_sharded
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("ShardedInference: torch.distributed is not initialised")
        self._aggregate = aggregate_sharded
        self.model, self.group = model, group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        n = g.num_nodes
        emb = model.embed_layer
        if n > emb.num_embeddings:
            raise RuntimeError("ShardedInference: the graph has %d nodes, the embedding %d rows"
                               % (n, emb.num_embeddings))
        self.bounds = shard_bounds(g.indptr, self.world) if bounds is None else check_bounds(bounds, n, self.world)
        self.lo, self.hi = self.bounds[self.rank], self.bounds[self.rank + 1]
        self.device = g.indptr.device
        mine = _parameter_digest(model)
        everyone = [None] * self.world
        dist.all_gather_object(everyone, mine, group=group)
        if any(d != everyone[0] for d in everyone):
            raise RuntimeError("ShardedInference: the ranks hold different parameters (digests %s)"
                               % ", ".join(d[:12] for d in everyone))
        e0, e1 = (int(x) for x in g.indptr[[self.lo, self.hi]].tolist())
        self.graph = CSRGraph(g.indptr[self.lo:self.hi + 1] - e0, g.indices[e0:e1])
        mean_agg_plan(self.graph)                                    # built once, kept with the shard
        self.width = max(max(l.in_feats, l.out_feats) for l in model.layers)
        self.cap_rows = max(self.bounds[r + 1] - self.bounds[r] for r in range(self.world))
        self.region_bytes = -(-max(self.cap_rows, 1) * self.width * 4 // 256) * 256
        self.own, self.opened, self.ptrs = dp.map_peer_buffers(3 * self.region_bytes, self.device, group,
                                                               "ShardedInference")
        self.agg = torch.empty((self.hi - self.lo) * self.width, dtype=torch.float32, device=self.device)
        self.token = torch.zeros(1, dtype=torch.float32, device=self.device)
        self.reading = set()          # regions peers may still read: read by an aggregation since the last barrier
        self.events = None            # a list: inference() appends (tag, recorded cuda.Event) at each phase

    # ---- regions ------------------------------------------------------------------------------------------
    def _blocks(self, region: int) -> List[int]:
        return [self.ptrs[r] + region * self.region_bytes for r in range(self.world)]

    def _own(self, region: int, F: int) -> torch.Tensor:
        rows = self.hi - self.lo
        if rows == 0:
            return torch.empty((0, F), dtype=torch.float32, device=self.device)
        return torch.as_tensor(_DeviceRegion(self.own + region * self.region_bytes, rows, F), device=self.device)

    def _barrier(self) -> None:
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(self.token, group=self.group)
        self.reading.clear()

    def _write(self, region: int) -> None:
        """Before this rank overwrites `region`: no peer may still be reading it."""
        if region in self.reading:
            self._barrier()

    def _mean(self, region: int, F: int) -> torch.Tensor:
        """Neighbour mean of this shard over every rank's rows of `region` ([rows][F] each)."""
        self._barrier()                                              # every rank's rows are written
        self._mark("barrier")
        rows = self.hi - self.lo
        out = self.agg[:rows * F].view(rows, F)
        self._aggregate(self.graph, self.bounds, self._blocks(region), F, out)
        self.reading.add(region)
        self._mark("aggregate")
        return out

    def _mark(self, tag: str) -> None:
        if self.events is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.events.append((tag, ev))

    def _own_rows(self) -> torch.Tensor:
        """Layer-0 input of this shard: SAGE._all_rows restricted to nodes [lo, hi)."""
        m, lo, rows = self.model, self.lo, self.hi - self.lo
        emb = m.embed_layer
        ids = torch.arange(lo, self.hi, device=self.device)
        if m.embed_name == "eff":
            return emb(ids)
        h = emb.rows_range(lo, rows)
        if h is not None:
            return h
        return emb(ids, torch.arange(rows + 1, device=self.device))

    @torch.no_grad()
    def inference(self) -> torch.Tensor:
        """[hi - lo, n_classes] logits of this shard's nodes: the function model.inference(g)[lo:hi] computes,
        in the operation order of SAGEConv.forward_full.  Collective."""
        layers = self.model.layers
        self._mark("start")
        cur, nxt = self._IN, self._OUT
        self._write(cur)
        if self.hi > self.lo:
            self._own(cur, layers[0].in_feats).copy_(self._own_rows())
        self._mark("rows")
        for l, layer in enumerate(layers):
            x = self._own(cur, layer.in_feats)
            if layer.in_feats > layer.out_feats:                    # fc_neigh before the mean
                self._write(self._PROJ)
                torch.mm(x, layer.fc_neigh.weight.t(), out=self._own(self._PROJ, layer.out_feats))
                self._mark("gemm")
                neigh = self._mean(self._PROJ, layer.out_feats)
            else:
                neigh = self._mean(cur, layer.in_feats)
                neigh = torch.mm(neigh, layer.fc_neigh.weight.t())
            self._write(nxt)
            out = self._own(nxt, layer.out_feats)
            torch.mm(x, layer.fc_self.weight.t(), out=out)
            out += neigh
            if layer.bias is not None:
                out += layer.bias
            if l != len(layers) - 1:
                torch.relu_(out)
            self._mark("gemm")
            cur, nxt = nxt, cur
        return self._own(cur, layers[-1].out_feats).clone()

    @torch.no_grad()
    def evaluate(self, labels: torch.Tensor, val_nid: torch.Tensor, test_nid: torch.Tensor):
        """(validation accuracy, test accuracy) of the sharded inference, the same numbers on every rank and
        the ones sage.evaluate computes: each rank marks the hits among its own nodes of each set, one
        all-reduce assembles the hit vectors, and the accuracy is taken over them as sage.evaluate does."""
        import torch.distributed as dist
        pred = self.inference().argmax(1)
        dev = self.device
        own_hit = pred == labels[self.lo:self.hi].to(dev)
        nids = [val_nid.to(dev), test_nid.to(dev)]
        hits = []
        for nid in nids:
            inside = (nid >= self.lo) & (nid < self.hi)
            h = torch.zeros(nid.numel(), dtype=torch.int32, device=dev)
            h[inside] = own_hit[nid[inside] - self.lo].to(torch.int32)
            hits.append(h)
        flat = torch.cat(hits)
        if self.world > 1:
            dist.all_reduce(flat, group=self.group)
        val_hit, test_hit = flat[:nids[0].numel()] != 0, flat[nids[0].numel():] != 0
        return float(val_hit.float().mean()), float(test_hit.float().mean())

    def close(self) -> None:
        """Collective: frees this rank's buffer once no rank reads it any more."""
        if self.own is None:
            return
        import torch.distributed as dist
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)
        dp.release_peer_buffers(self.own, self.opened)
        self.own, self.opened, self.agg = None, [], None


def _parameter_digest(model: SAGE) -> str:
    """sha256 of the dense layers and the TT cores, in a fixed order."""
    import hashlib
    h = hashlib.sha256()
    for t in list(model.dense_parameters()) + list(model.embed_layer.tt_cores):
        h.update(t.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


def synthetic_graph(num_nodes: int, num_edges: int, device, seed: int = 0, alpha: float = 2.1
                    ) -> CSRGraph:
    """Power-law in-degrees (Pareto tail `alpha`, rescaled to `num_edges` in total, at least one
    in-edge per node), uniformly random in-neighbours; int64 indptr, int32 indices."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    u = torch.rand(num_nodes, generator=g, device=device, dtype=torch.float64)
    w = (1.0 - u).clamp_min(1e-12).pow(-1.0 / alpha)
    w = w.clamp_max(float(num_nodes) ** 0.5 * 10.0)
    deg = torch.floor(w * (num_edges - num_nodes) / w.sum()).to(torch.int64) + 1
    short = int(num_edges - int(deg.sum()))
    if short > 0:   # hand the rounding remainder to the first nodes
        deg[:short] += 1
    indptr = torch.zeros(num_nodes + 1, dtype=torch.int64, device=device)
    torch.cumsum(deg, 0, out=indptr[1:])
    indices = torch.randint(0, num_nodes, (int(indptr[-1]),), generator=g, device=device,
                            dtype=torch.int32)
    return CSRGraph(indptr, indices)


def synthetic_community_graph(num_nodes: int, num_edges: int, k: int, p_in: float, device,
                              seed: int = 0, ordered: bool = False):
    """Symmetric graph with k equal communities (an undirected edge stays inside its community
    with probability p_in) whose node ids are scrambled -- what a raw dataset looks like before
    graphloader.py:399-454 reorders it; ordered=True keeps the ids community by community, i.e. the graph
    AFTER a METIS-k reorder (BASELINE config 3).  Returns (graph, community id of every node)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    half = num_edges // 2
    size = (num_nodes + k - 1) // k
    src = torch.randint(0, num_nodes, (half,), generator=g, device=device)
    inside = torch.rand(half, generator=g, device=device) < p_in
    lo = (src // size) * size
    width = torch.minimum(torch.full_like(lo, size), num_nodes - lo)
    near = lo + (torch.rand(half, generator=g, device=device, dtype=torch.float64) * width).long()
    far = torch.randint(0, num_nodes, (half,), generator=g, device=device)
    dst = torch.where(inside, near, far)
    scramble = (torch.arange(num_nodes, device=device) if ordered
                else torch.randperm(num_nodes, generator=g, device=device))
    s, d = scramble[torch.cat([src, dst])], scramble[torch.cat([dst, src])]
    order = torch.sort(d * num_nodes + s).indices
    s, d = s[order], d[order]
    indptr = torch.zeros(num_nodes + 1, dtype=torch.int64, device=device)
    torch.cumsum(torch.bincount(d, minlength=num_nodes), 0, out=indptr[1:])
    comm = torch.empty(num_nodes, dtype=torch.int64, device=device)
    comm[scramble] = torch.arange(num_nodes, device=device) // size
    return CSRGraph(indptr, s.to(torch.int32)), comm


class Trainer:
    """One optimisation step of the reference's training loop (sage_dgl_partition.py:205-262):
    Adam on the SAGE layers, the TT cores by their fused SGD (single GPU, --sparse) or -- data
    parallel -- by the exchange step of dp.py: the dense layers' gradients live in ONE flat buffer
    (the parameters' .grad are views of it) that is all-reduced in place, the TT cores go through
    dp.PeerExchange (gradient exchange + update in one kernel over NVLink peer memory) when the
    ranks share a node, else through the same all-reduce followed by ttg_apply_optimizer."""

    def __init__(self, model: SAGE, lr: float = 0.003, world: int = 1, peer_exchange: bool = True):
        self.model, self.world = model, world
        self.opt = torch.optim.Adam(model.dense_parameters(), lr=lr)
        self.flat = None
        self.xchg = None
        if world > 1:
            model.embed_layer.sparse = False
            params = model.dense_parameters()
            self.flat = torch.zeros(sum(p.numel() for p in params), dtype=torch.float32,
                                    device=params[0].device)
            off = 0
            for p in params:      # autograd accumulates into an existing .grad in place
                p.grad = self.flat[off:off + p.numel()].view_as(p)
                off += p.numel()
            if peer_exchange:
                # PeerExchange is collective and agrees on success over the group: either every rank has it
                # or every rank raised (and freed its buffers) -> all fall back to NCCL together
                try:
                    self.xchg = dp.PeerExchange(model.embed_layer.tt_cores)
                except RuntimeError:
                    self.xchg = None          # not one node / no peer access: NCCL for the cores too
        self.steps = 0
        self.check_every = 64                 # steps between looks at the exchange kernel's error word

    def step(self, blocks, input_nodes, labels) -> torch.Tensor:
        m = self.model
        logits = m(blocks, input_nodes)
        loss = F.cross_entropy(logits, labels)
        if self.world == 1:
            self.opt.zero_grad(set_to_none=True)
            loss.backward()
        else:
            emb = m.embed_layer
            self.flat.zero_()
            loss.backward()
            cores = [c.grad for c in emb.tt_cores]
            dp.allreduce_mean([self.flat])          # in place: the .grad views see the mean
            if self.xchg is not None:
                self.xchg.step(cores, list(emb.tt_cores), "sgd", emb.learning_rate)
            else:
                reduced = dp.allreduce_mean(cores)  # in place too (tt_dense_backward's flat buffer)
                dp.apply_optimizer(emb.tt_p_shapes, emb.tt_q_shapes, emb.tt_ranks, list(emb.tt_cores),
                                   [gr.contiguous() for gr in reduced], emb.learning_rate)
            for c in emb.tt_cores:
                c.grad = None
        self.opt.step()
        self.steps += 1
        if self.xchg is not None and self.steps % self.check_every == 0 and self.xchg.failed_epoch():
            raise RuntimeError("Trainer: a peer did not arrive at exchange step %d; the update of that step "
                               "was skipped on this rank, the replicas may have diverged"
                               % self.xchg.failed_epoch())
        return loss

    def failed_epoch(self) -> int:
        return self.xchg.failed_epoch() if self.xchg is not None else 0

    def close(self) -> None:
        if self.xchg is not None:
            self.xchg.close()
            self.xchg = None
