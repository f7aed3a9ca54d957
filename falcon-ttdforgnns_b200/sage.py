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
from gnn_ops import Block, SAGEConv
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
