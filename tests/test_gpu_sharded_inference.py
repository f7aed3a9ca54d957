"""Sharded full-neighbour inference (csrc/spmm.cu ttg_mean_agg_sharded, gnn_ops.aggregate_sharded,
sage.ShardedInference).  The kernel runs on one GPU with 1 .. 8 "virtual peers" -- row blocks that are separate
allocations -- and must give the bits of ttg_mean_agg on the concatenated rows.  ShardedInference runs under a
one-rank process group here and on two GPUs in a torchrun worker (tests/sharded_inference_worker.py)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5                    # the inference bar of tests/test_gpu_sage_inference.py
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "sharded_inference_worker.py")


def rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-300))


def _graph(indptr, indices):
    from sampler import CSRGraph
    return CSRGraph(indptr.to(DEV, torch.int64).contiguous(), indices.to(DEV, torch.int32).contiguous())


def _sharded_mean(g, x, bounds):
    """Every shard's mean over blocks that are separate allocations, concatenated."""
    from gnn_ops import aggregate_sharded
    from sampler import CSRGraph
    W = len(bounds) - 1
    blocks = [x[bounds[r]:bounds[r + 1]].clone() for r in range(W)]
    ptrs = [b.data_ptr() if b.numel() else 0 for b in blocks]
    outs = []
    for r in range(W):
        lo, hi = bounds[r], bounds[r + 1]
        e0, e1 = int(g.indptr[lo]), int(g.indptr[hi])
        shard = CSRGraph(g.indptr[lo:hi + 1] - e0, g.indices[e0:e1])
        out = torch.full((hi - lo, x.size(1)), float("nan"), device=DEV)
        outs.append(aggregate_sharded(shard, bounds, ptrs, x.size(1), out))
    return torch.cat(outs)


def _uneven(n, W, gen):
    """W + 1 bounds from 0 to n with uneven shards: the first one empty at W = 2, the second from W = 3 on."""
    cuts = sorted(torch.randint(0, n + 1, (W - 1,), generator=gen).tolist())
    b = [0] + cuts + [n]
    if W == 2:
        b[1] = 0
    elif W > 2:
        b[2] = b[1]
    assert b[0] == 0 and b[-1] == n and all(b[r] <= b[r + 1] for r in range(W))
    return b


@pytest.mark.parametrize("F", [1, 47, 100, 256, 260])
def test_virtual_peers_give_the_bits_of_the_whole_graph_mean(ttg_lib, F):
    import sage
    from gnn_ops import aggregate_full
    g = sage.synthetic_graph(30_000, 900_000, torch.device(DEV), seed=11)
    deg = g.indptr[1:] - g.indptr[:-1]
    assert int(deg.max()) > 4 * 256                    # rows of several work items: the finalize pass runs
    gen = torch.Generator().manual_seed(F)
    x = torch.randn((g.num_nodes, F), generator=gen).to(DEV)
    want = aggregate_full(g, x)
    for W in range(1, 9):
        for bounds in (sage.shard_bounds(g.indptr, W), _uneven(g.num_nodes, W, gen)):
            got = _sharded_mean(g, x, bounds)
            assert torch.equal(got, want), (F, W, bounds)


@pytest.mark.parametrize("F", [47, 256])
def test_every_edge_crosses_shards(ttg_lib, F):
    """Four shards, every in-neighbour of a node lives in another shard; a quarter of the nodes have none."""
    from gnn_ops import aggregate_full
    n, W = 8000, 4
    bounds = [0, 1000, 3000, 3001, 8000]
    gen = torch.Generator().manual_seed(4)
    owner = torch.bucketize(torch.arange(n), torch.tensor(bounds[1:-1]), right=True)
    deg = torch.randint(0, 700, (n,), generator=gen)
    deg[torch.randperm(n, generator=gen)[:n // 4]] = 0
    indptr = torch.zeros(n + 1, dtype=torch.int64)
    indptr[1:] = torch.cumsum(deg, 0)
    src = torch.randint(0, n, (int(indptr[-1]),), generator=gen)
    dst = torch.repeat_interleave(torch.arange(n), deg)
    same = owner[src] == owner[dst]
    src[same] = (src[same] + 3001) % n                 # leave the shard of the destination
    while bool((owner[src] == owner[dst]).any()):
        same = owner[src] == owner[dst]
        src[same] = (src[same] + 997) % n
    g = _graph(indptr, src.to(torch.int32))
    x = torch.randn((n, F), generator=gen).to(DEV)
    got = _sharded_mean(g, x, bounds)
    assert torch.equal(got, aggregate_full(g, x))
    assert bool((got[(deg == 0).to(DEV)] == 0).all())


def test_graph_without_edges(ttg_lib):
    g = _graph(torch.zeros(301, dtype=torch.int64), torch.zeros(0, dtype=torch.int32))
    for F in (3, 128):
        got = _sharded_mean(g, torch.randn((300, F), device=DEV), [0, 100, 100, 300])
        assert got.shape == (300, F) and bool((got == 0).all())


# ---- ShardedInference under a one-rank process group ----------------------------------------------------------
N_NODES = 20_000


def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.fixture
def one_rank():
    import torch.distributed as dist
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % _free_port(), rank=0, world_size=1)
    try:
        yield
    finally:
        dist.destroy_process_group()


def _model(kind, seed=3):
    import sage
    torch.manual_seed(seed)
    m = sage.SAGE(N_NODES, 100, 128, 7, 3, 0.5, (16, 16), (28, 28, 28), (4, 5, 5), sparse=True,
                  learning_rate=0.05, embed_name=kind).to(DEV)
    with torch.no_grad():            # rows of order 1e-2 instead of 1e-6
        for c in m.embed_layer.tt_cores:
            c.mul_(8.0 if kind != "eff" else 1.0)
    return m


@pytest.mark.parametrize("kind", ["fbtt", "eff"])
def test_one_rank_matches_inference_and_evaluate(ttg_lib, one_rank, kind):
    import sage
    g = sage.synthetic_graph(N_NODES, 600_000, torch.device(DEV), seed=4)
    m = _model(kind)
    labels = torch.randint(0, 7, (N_NODES,), generator=torch.Generator().manual_seed(5)).to(DEV)
    perm = torch.randperm(N_NODES, generator=torch.Generator().manual_seed(6)).to(DEV)
    val_nid, test_nid = perm[:5000], perm[5000:9000]
    before = [p.detach().clone() for p in m.embed_layer.tt_cores] + [p.detach().clone() for p in m.dense_parameters()]
    flags = [mod.training for mod in m.modules()]
    inf = sage.ShardedInference(m, g)
    try:
        assert inf.bounds == [0, N_NODES] and (inf.lo, inf.hi) == (0, N_NODES)
        got = inf.inference()
        again = inf.inference()
        val, test = inf.evaluate(labels, val_nid, test_nid)
    finally:
        inf.close()
    torch.cuda.synchronize()
    after = [p.detach() for p in m.embed_layer.tt_cores] + [p.detach() for p in m.dense_parameters()]
    assert all(torch.equal(a, b) for a, b in zip(after, before))
    assert [mod.training for mod in m.modules()] == flags
    assert all(p.grad is None for p in m.parameters())
    want = m.inference(g)
    assert got.shape == want.shape and rel(got, want) < TOL
    assert torch.equal(got.argmax(1), want.argmax(1))
    assert torch.equal(got, again)
    val_ref, test_ref, _ = sage.evaluate(m, g, labels, val_nid, test_nid)
    assert (val, test) == (val_ref, test_ref)


def test_one_rank_refusals(ttg_lib, one_rank):
    import sage
    m = _model("fbtt")
    big = sage.synthetic_graph(N_NODES + 1, 100_000, torch.device(DEV), seed=1)
    with pytest.raises(RuntimeError, match="embedding"):
        sage.ShardedInference(m, big)
    g = sage.synthetic_graph(N_NODES, 100_000, torch.device(DEV), seed=1)
    for bad in ([0, N_NODES - 1], [1, N_NODES], [0, 5, N_NODES]):
        with pytest.raises(ValueError):
            sage.ShardedInference(m, g, bounds=bad)
    inf = sage.ShardedInference(m, g, bounds=[0, N_NODES])   # what was refused left nothing behind
    inf.close()


# ---- two GPUs ---------------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_read_each_other_over_nvlink(ttg_lib):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), WORKER]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "SHARDED_INFERENCE_OK" in r.stdout
