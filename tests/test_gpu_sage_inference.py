"""Full-neighbour evaluation of GraphSAGE: the whole-graph mean aggregation (gnn_ops.aggregate_full, csrc/spmm.cu
ttg_mean_agg) against a float64 index_add mean, SAGE.inference against a float64 restatement and against the
training path, and an end-to-end check that sage.Trainer learns what sage.evaluate then measures.  Tolerance:
1e-5 relative to the tensor's maximum."""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5


def rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-300))


def _graph(indptr, indices):
    from sampler import CSRGraph
    return CSRGraph(indptr.to(DEV, torch.int64).contiguous(), indices.to(DEV, torch.int32).contiguous())


def _mean64(g, x):
    """float64 mean over the in-neighbours (index_add), 0 rows where there are none."""
    n = g.num_nodes
    deg = (g.indptr[1:] - g.indptr[:-1])
    dst = torch.repeat_interleave(torch.arange(n, device=DEV), deg)
    out = torch.zeros((n, x.size(1)), dtype=torch.float64, device=DEV)
    out.index_add_(0, dst, x.double()[g.indices.long()])
    return out / deg.clamp(min=1).double().unsqueeze(1)


def _check(g, F, seed=0):
    from gnn_ops import aggregate_full
    gen = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn((g.num_nodes, F), generator=gen, device=DEV)
    got = aggregate_full(g, x)
    torch.cuda.synchronize()
    want = _mean64(g, x)
    assert got.shape == (g.num_nodes, F) and got.dtype == torch.float32
    assert rel(got, want) < TOL, (F, rel(got, want))
    return x, got


# ---- 1. the kernel ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("F", [1, 3, 47, 100, 128, 256])
def test_power_law_graph(ttg_lib, F):
    import sage
    g = sage.synthetic_graph(50_000, 2_500_000, torch.device(DEV), seed=1)
    deg = g.indptr[1:] - g.indptr[:-1]
    assert int(deg.max()) > 4 * 256          # rows of several work items
    _check(g, F)


@pytest.mark.parametrize("F", [47, 256])
def test_star_with_isolated_nodes(ttg_lib, F):
    """Node 3 has 200,003 in-edges (782 work items); every other node has none."""
    n, hub, e = 1000, 3, 200_003
    deg = torch.zeros(n, dtype=torch.int64)
    deg[hub] = e
    indptr = torch.zeros(n + 1, dtype=torch.int64)
    indptr[1:] = torch.cumsum(deg, 0)
    indices = torch.randint(0, n, (e,), generator=torch.Generator().manual_seed(5), dtype=torch.int32)
    g = _graph(indptr, indices)
    _, got = _check(g, F)
    others = torch.ones(n, dtype=torch.bool, device=DEV)
    others[hub] = False
    assert bool((got[others] == 0).all())


def test_zero_degree_destinations_are_exact_zero_rows(ttg_lib):
    gen = torch.Generator().manual_seed(9)
    n = 5000
    deg = torch.randint(0, 600, (n,), generator=gen)
    deg[torch.randperm(n, generator=gen)[:1500]] = 0
    indptr = torch.zeros(n + 1, dtype=torch.int64)
    indptr[1:] = torch.cumsum(deg, 0)
    indices = torch.randint(0, n, (int(indptr[-1]),), generator=gen, dtype=torch.int32)
    g = _graph(indptr, indices)
    for F in (47, 100):
        x = torch.full((n, F), float("nan"), device=DEV)   # NaN rows nobody reads
        used = torch.zeros(n, dtype=torch.bool, device=DEV)
        used[g.indices.long()] = True
        x[used] = torch.randn((int(used.sum()), F), device=DEV)
        from gnn_ops import aggregate_full
        got = aggregate_full(g, x)
        zero = (deg == 0).to(DEV)
        assert bool((got[zero] == 0).all()) and not bool(torch.signbit(got[zero]).any())
        assert rel(got[~zero], _mean64(g, torch.nan_to_num(x))[~zero]) < TOL


def test_graph_without_edges(ttg_lib):
    from gnn_ops import aggregate_full
    g = _graph(torch.zeros(301, dtype=torch.int64), torch.zeros(0, dtype=torch.int32))
    for F in (3, 128):
        out = aggregate_full(g, torch.randn((300, F), device=DEV))
        assert out.shape == (300, F) and bool((out == 0).all())


def test_single_node(ttg_lib):
    from gnn_ops import aggregate_full
    x = torch.randn((1, 47), device=DEV)
    g = _graph(torch.tensor([0, 0]), torch.zeros(0, dtype=torch.int32))
    assert bool((aggregate_full(g, x) == 0).all())
    g = _graph(torch.tensor([0, 700]), torch.zeros(700, dtype=torch.int32))   # a self loop, 700 times
    for F in (47, 256):
        x = torch.randn((1, F), device=DEV)
        assert rel(aggregate_full(g, x), x) < TOL


# ---- 2. determinism ---------------------------------------------------------------------------------------
def test_same_bits_from_every_call_and_width(ttg_lib):
    import sage
    from gnn_ops import aggregate, aggregate_full, Block
    g = sage.synthetic_graph(50_000, 2_500_000, torch.device(DEV), seed=2)
    gen = torch.Generator(device=DEV).manual_seed(3)
    x256 = torch.randn((g.num_nodes, 256), generator=gen, device=DEV)
    x47 = torch.randn((g.num_nodes, 47), generator=gen, device=DEV)
    a = aggregate_full(g, x256)
    plan = g._mean_agg_plan[1]
    b = aggregate_full(g, x47)
    c = aggregate_full(g, x256)
    d = aggregate_full(g, x47)
    assert g._mean_agg_plan[1] is plan                     # one plan for every width
    assert torch.equal(a, c) and torch.equal(b, d)
    fresh = sage.synthetic_graph(50_000, 2_500_000, torch.device(DEV), seed=2)   # its own plan
    assert torch.equal(aggregate_full(fresh, x47), b)
    # rows of one work item sum in edge order, as the one-warp-per-destination kernel does: same bits
    deg = g.indptr[1:] - g.indptr[:-1]
    short = deg <= 256
    with torch.no_grad():
        old = aggregate(Block(g.indptr, g.indices, g.num_nodes, g.num_nodes), x256, mean=True)
    assert torch.equal(old[short], a[short])
    assert rel(a, old) < TOL


# ---- 3.-5. SAGE.inference ---------------------------------------------------------------------------------
N_NODES = 20_000


def _model(kind, fuse_input=False, seed=3):
    import sage
    torch.manual_seed(seed)
    m = sage.SAGE(N_NODES, 100, 128, 7, 3, 0.5, (16, 16), (28, 28, 28), (4, 5, 5), sparse=True,
                  learning_rate=0.05, embed_name="eff" if kind == "eff" else "fbtt", fuse_input=fuse_input).to(DEV)
    with torch.no_grad():            # rows of order 1e-2 instead of 1e-6
        for c in m.embed_layer.tt_cores:
            c.mul_(8.0 if kind != "eff" else 1.0)
    if kind == "fbtt_lookup":        # the lookup on arange(N) instead of the row kernel on the implicit range
        m.embed_layer.rows_range = lambda first, num: None
    return m


def _rows64(emb, n):
    """Rows 0 .. n - 1 of the TT table in float64 (tt_matrix_to_full contracts the same way but returns fp32)."""
    from FBTT.tt_embeddings_ops import tt_matrix_to_full
    p, q, r = emb.tt_p_shapes, emb.tt_q_shapes, emb.tt_ranks
    c = [emb.tt_cores[t].detach().double().reshape(p[t], r[t], q[t], r[t + 1]) for t in range(3)]
    full = torch.einsum("aiqj,bjrk,cksl->abcqrs", *c).reshape(p[0] * p[1] * p[2], q[0] * q[1] * q[2])
    ref32 = tt_matrix_to_full(p, q, r, [t.detach() for t in emb.tt_cores], [1, 0, 2, 3])
    assert rel(ref32, full) < 1e-6            # same row and column order
    return full[:n]


def _inference64(m, g):
    h = _rows64(m.embed_layer, g.num_nodes)
    for l, layer in enumerate(m.layers):
        ws, wn = layer.fc_self.weight.detach().double(), layer.fc_neigh.weight.detach().double()
        h = h @ ws.t() + _mean64(g, h) @ wn.t() + layer.bias.detach().double()
        if l != len(m.layers) - 1:
            h = torch.relu(h)
    return h


@pytest.mark.parametrize("kind", ["fbtt", "fbtt_lookup", "eff"])
def test_inference_against_float64(ttg_lib, kind):
    import sage
    g = sage.synthetic_graph(N_NODES, 600_000, torch.device(DEV), seed=4)
    m = _model(kind)
    assert m.layers[0].in_feats <= m.layers[0].out_feats and m.layers[2].in_feats > m.layers[2].out_feats
    m.eval()
    got = m.inference(g)
    assert got.shape == (N_NODES, 7) and not got.requires_grad
    assert rel(got, _inference64(m, g)) < TOL


def _bounded_graph(n, max_deg, seed):
    gen = torch.Generator().manual_seed(seed)
    deg = torch.randint(0, max_deg + 1, (n,), generator=gen)
    indptr = torch.zeros(n + 1, dtype=torch.int64)
    indptr[1:] = torch.cumsum(deg, 0)
    indices = torch.randint(0, n, (int(indptr[-1]),), generator=gen, dtype=torch.int32)
    return _graph(indptr, indices)


@pytest.mark.parametrize("fuse_input", [False, True])
def test_inference_equals_training_path(ttg_lib, fuse_input):
    """In-degrees <= 32: NeighborSampler([32, 32, 32]) takes every in-edge, so the eval-mode forward on the
    sampled blocks computes the same function as the whole-graph inference."""
    import sampler
    g = _bounded_graph(N_NODES, 32, 6)
    m = _model("fbtt", fuse_input=fuse_input)
    assert m.fuse_input == fuse_input
    seeds = torch.randperm(N_NODES, generator=torch.Generator().manual_seed(7))[:1024].to(DEV)
    inp, outp, blocks = sampler.NeighborSampler([32, 32, 32]).sample_blocks(g, seeds, seed=13)
    for blk in blocks:
        assert blk.indices.numel() == int((g.indptr[1:] - g.indptr[:-1])[inp[:blk.num_dst]].sum())
    m.eval()
    with torch.no_grad():
        want = m(blocks, inp)
    full = m.inference(g)
    assert rel(full[seeds], want) < TOL
    other = _model("fbtt", fuse_input=not fuse_input)         # same seed: same weights
    other.eval()
    assert torch.equal(other.inference(g), full)             # fuse_input plays no part


@pytest.mark.parametrize("kind", ["fbtt", "fbtt_lookup", "eff"])
@pytest.mark.parametrize("training", [True, False])
def test_inference_changes_nothing(ttg_lib, kind, training):
    import sage
    g = sage.synthetic_graph(N_NODES, 300_000, torch.device(DEV), seed=8)
    m = _model(kind)
    m.train(training)
    before = copy.deepcopy([p.detach().clone() for p in m.embed_layer.tt_cores] +
                           [p.detach().clone() for p in m.dense_parameters()])
    flags = [mod.training for mod in m.modules()]
    first = m.inference(g)
    second = m.inference(g)
    torch.cuda.synchronize()
    after = [p.detach() for p in m.embed_layer.tt_cores] + [p.detach() for p in m.dense_parameters()]
    assert all(torch.equal(a, b) for a, b in zip(after, before))
    assert [mod.training for mod in m.modules()] == flags and m.training == training
    assert torch.equal(first, second)
    assert all(p.grad is None for p in m.parameters())


# ---- 6. the stack learns ----------------------------------------------------------------------------------
LEARN_STEPS = 100
LEARN_MIN_ACC = 0.56          # chance (0.125) plus half the measured margin (0.9995 - 0.125)
LEARN_TT_LR = 0.2
LEARN_CORE_SCALE = 20.0


def test_training_then_evaluate_learns_communities(ttg_lib):
    """8 communities of 2,500 nodes, 90% of the edges inside; the label of a node is its community, its input
    is its TT embedding row (learnt).  Before training the full-neighbour evaluation is at chance (1/8);
    after LEARN_STEPS Trainer steps of 1,024 seeds with fanouts [5, 10, 15] it must clear LEARN_MIN_ACC on
    both the validation and the test nodes.  Measured on a B200: 0.126 / 0.128 before training; 0.9465 /
    0.9475 after 50 steps, 0.9995 / 0.9995 after 100 (validation / test), 0.23 s of training."""
    import sage
    import sampler
    dev = torch.device(DEV)
    k, n = 8, 20_000
    g, comm = sage.synthetic_community_graph(n, 400_000, k, 0.9, dev, seed=1)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(2)).to(DEV)
    train_nid, val_nid, test_nid = perm[:12_000], perm[12_000:16_000], perm[16_000:]
    torch.manual_seed(0)
    m = sage.SAGE(n, 100, 128, k, 3, 0.0, (16, 16), (28, 28, 28), (4, 5, 5), sparse=True,
                  learning_rate=LEARN_TT_LR, embed_name="fbtt").to(DEV)
    with torch.no_grad():
        for c in m.embed_layer.tt_cores:
            c.mul_(LEARN_CORE_SCALE)
    val0, test0, pred0 = sage.evaluate(m, g, comm, val_nid, test_nid)
    assert m.training and pred0.shape == (n, k)
    assert abs(val0 - 1 / k) < 0.08 and abs(test0 - 1 / k) < 0.08, (val0, test0)
    trainer = sage.Trainer(m, lr=0.01)
    smp = sampler.NeighborSampler([5, 10, 15])
    gen = torch.Generator().manual_seed(3)
    for step in range(LEARN_STEPS):
        seeds = train_nid[torch.randint(0, train_nid.numel(), (1024,), generator=gen).to(DEV)]
        seeds = torch.unique(seeds)
        inp, outp, blocks = smp.sample_blocks(g, seeds, seed=step)
        trainer.step(blocks, inp, comm[outp])
    val1, test1, _ = sage.evaluate(m, g, comm, val_nid, test_nid)
    print("accuracy before %.4f / %.4f, after %d steps %.4f / %.4f" % (val0, test0, LEARN_STEPS, val1, test1))
    assert val1 > LEARN_MIN_ACC and test1 > LEARN_MIN_ACC, (val1, test1)

