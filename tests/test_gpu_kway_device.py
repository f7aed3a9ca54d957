"""The multilevel k-way partitioner on the device (csrc/kway.cu, reorder.kway_partition_device) against the bars
tests/test_partition_cpu.py sets for the host partitioner: balance bounds, cut against known optima and planted
partitions, determinism in the seed, edge cases, argument checks; reorder_graph(g, "kway") and its composition."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import reorder_oracle as ro

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _csr(n, src, dst):
    """in-neighbour lists: row dst holds src"""
    order = np.argsort(dst, kind="stable")
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(dst, minlength=n), out=indptr[1:])
    return indptr, np.ascontiguousarray(src[order], dtype=np.int32)


def _grid(w, h):
    ids = np.arange(w * h).reshape(h, w)
    a = np.concatenate([ids[:, :-1].ravel(), ids[:-1, :].ravel()])
    b = np.concatenate([ids[:, 1:].ravel(), ids[1:, :].ravel()])
    return _csr(w * h, np.concatenate([a, b]), np.concatenate([b, a]))


def _planted(rng, n, k, deg_in, deg_out):
    """k equal communities under scrambled ids: deg_in edges per node inside, deg_out anywhere"""
    lab = rng.permutation(n) % k
    src, dst = [], []
    for p in range(k):
        m = np.nonzero(lab == p)[0]
        src.append(rng.choice(m, size=m.shape[0] * deg_in // 2))
        dst.append(rng.choice(m, size=m.shape[0] * deg_in // 2))
    src.append(rng.integers(0, n, size=n * deg_out // 2))
    dst.append(rng.integers(0, n, size=n * deg_out // 2))
    s, d = np.concatenate(src), np.concatenate(dst)
    s, d = np.concatenate([s, d]), np.concatenate([d, s])
    indptr, indices = _csr(n, s, d)
    return indptr, indices, lab, int((lab[s] != lab[d]).sum())


def _community_graph(rng, n, k, deg, p_in):
    """tests/test_gpu_reorder.py's generator: k equal communities with scrambled ids; symmetric edges."""
    comm = rng.permutation(n) % k
    members = [np.nonzero(comm == c)[0] for c in range(k)]
    src = np.repeat(np.arange(n), deg)
    inside = rng.random(src.shape[0]) < p_in
    dst = rng.integers(0, n, size=src.shape[0])
    for c in range(k):
        sel = np.nonzero(inside & (comm[src] == c))[0]
        dst[sel] = members[c][rng.integers(0, members[c].shape[0], size=sel.shape[0])]
    s = np.concatenate([src, dst])
    d = np.concatenate([dst, src])
    order = np.lexsort((s, d))
    s, d = s[order], d[order]
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(d, minlength=n), out=indptr[1:])
    return indptr, s.astype(np.int32), comm


def _cut(indptr, indices, part):
    dst = np.repeat(np.arange(indptr.shape[0] - 1), np.diff(indptr))
    return int((part[dst] != part[indices]).sum())


def _bound(n, k, ub):
    ideal = -(-n // k)
    return max(ideal, int(ub * ideal))


def _floor_bound(n, k, ub):
    return int((n // k) / ub)


def _graph(indptr, indices):
    from sampler import CSRGraph
    return CSRGraph(torch.from_numpy(indptr).to(DEV), torch.from_numpy(indices).to(DEV))


def _kway(indptr, indices, k, ub=1.03, seed=0):
    import reorder
    part, cut = reorder.kway_partition_device(_graph(indptr, indices), k, ubfactor=ub, seed=seed, return_cut=True)
    assert part.dtype == torch.int32 and part.device.type == "cuda"
    return part.cpu().numpy(), cut


def _assert_balanced(part, n, k, ub=1.03):
    sizes = np.bincount(part, minlength=k)
    assert part.min() >= 0 and part.max() < k
    assert sizes.max() <= _bound(n, k, ub), (sizes.max(), _bound(n, k, ub))
    assert sizes.min() >= _floor_bound(n, k, ub), (sizes.min(), _floor_bound(n, k, ub))


@pytest.mark.parametrize("k", [2, 4, 16, 64])
def test_grid_parts_are_balanced_and_compact(ttg_lib, k):
    indptr, indices = _grid(64, 64)
    part, cut = _kway(indptr, indices, k)
    _assert_balanced(part, 4096, k)
    assert cut == _cut(indptr, indices, part)
    optimum = 2 * 64 if k == 2 else 2 * 2 * 64 * (int(round(k ** 0.5)) - 1)
    assert cut <= 2.0 * optimum, (cut, optimum)


def test_planted_communities_are_recovered(ttg_lib):
    rng = np.random.default_rng(0)
    n, k = 20000, 50
    indptr, indices, lab, planted_cut = _planted(rng, n, k, 12, 2)
    part, cut = _kway(indptr, indices, k)
    _assert_balanced(part, n, k)
    assert cut <= 1.02 * planted_cut, (cut, planted_cut)
    purity = np.mean([np.bincount(part[lab == c]).max() / float((lab == c).sum()) for c in range(k)])
    assert purity > 0.97


def test_deterministic_in_the_seed(ttg_lib):
    rng = np.random.default_rng(1)
    indptr, indices, _, _ = _planted(rng, 6000, 12, 8, 3)
    a, cut_a = _kway(indptr, indices, 12, seed=5)
    b, cut_b = _kway(indptr, indices, 12, seed=5)
    assert np.array_equal(a, b) and cut_a == cut_b
    c, _ = _kway(indptr, indices, 12, seed=6)
    _assert_balanced(c, 6000, 12)


def test_power_law_graph_beats_the_id_order_and_keeps_the_bound(ttg_lib):
    rng = np.random.default_rng(2)
    n, m = 30000, 4
    targets = np.empty((n, m), dtype=np.int64)
    pool = list(range(m))
    for v in range(m, n):
        pick = rng.integers(0, len(pool), size=m)
        targets[v] = [pool[i] for i in pick]
        pool.extend(targets[v].tolist())
        pool.extend([v] * m)
    src = np.repeat(np.arange(m, n), m)
    dst = targets[m:].ravel()
    indptr, indices = _csr(n, np.concatenate([src, dst]), np.concatenate([dst, src]))
    k = 25
    part, cut = _kway(indptr, indices, k, ub=1.05)
    _assert_balanced(part, n, k, 1.05)
    blocks = np.arange(n) // (n // k)
    assert cut < 0.8 * _cut(indptr, indices, blocks)


def test_directed_cliques_self_loops_duplicates_and_isolated_nodes(ttg_lib):
    edges = [(a, b) for a in range(4) for b in range(4) if a < b] + \
            [(a, b) for a in range(4, 8) for b in range(4, 8) if a < b] + [(3, 4), (2, 2), (0, 1)]
    src = np.array([e[0] for e in edges])
    dst = np.array([e[1] for e in edges])
    indptr, indices = _csr(9, src, dst)
    part, cut = _kway(indptr, indices, 2, ub=1.2)
    assert len(set(part[:4])) == 1 and len(set(part[4:8])) == 1 and part[0] != part[4]
    assert cut == 1
    assert np.bincount(part, minlength=2).max() <= 5


def test_edge_cases(ttg_lib):
    indptr, indices = _grid(8, 8)
    part, cut = _kway(indptr, indices, 1)
    assert not part.any() and cut == 0
    part, cut = _kway(indptr, indices, 64)                    # k = N: one node per part
    assert sorted(part.tolist()) == list(range(64)) and cut == indices.shape[0]
    empty = np.zeros(6, dtype=np.int64)                       # five nodes, no edges
    part, cut = _kway(empty, np.zeros(0, dtype=np.int32), 3)
    assert cut == 0 and np.bincount(part, minlength=3).max() <= 2
    part, cut = _kway(np.zeros(1, dtype=np.int64), np.zeros(0, dtype=np.int32), 1)   # no nodes
    assert part.size == 0 and cut == 0


def test_reported_cut_is_a_recount(ttg_lib):
    rng = np.random.default_rng(4)
    indptr, indices, _, _ = _planted(rng, 5000, 10, 6, 4)
    part, cut = _kway(indptr, indices, 10, seed=3)
    assert cut == _cut(indptr, indices, part)


def test_reorder_graph_kway_sorts_part_by_part(ttg_lib):
    import reorder
    rng = np.random.default_rng(5)
    indptr, indices, _ = _community_graph(rng, 3000, 6, 8, 0.9)
    g = _graph(indptr, indices)
    g2, perm = reorder.reorder_graph(g, "kway", k=6, seed=2)
    part = reorder.kway_partition_device(g, 6, seed=2).cpu().numpy()
    p = perm.cpu().numpy()
    assert np.array_equal(p, np.argsort(part, kind="stable"))
    ip, ix, _ = ro.permute_csr(indptr, indices, p)
    assert np.array_equal(g2.indptr.cpu().numpy(), ip)
    assert np.array_equal(g2.indices.cpu().numpy(), ix)


def test_recursive_reorder_composes_the_permutations(ttg_lib):
    import reorder
    rng = np.random.default_rng(6)
    indptr, indices, _ = _community_graph(rng, 4000, 8, 8, 0.9)
    g = _graph(indptr, indices)
    g_final, perm = reorder.recursive_metis_reorder(g, [4, 6, 12], algo="kway")
    cur, total = g, np.arange(4000)
    for level, k in enumerate([4, 6, 12]):
        cur, p = reorder.reorder_graph(cur, "kway", k=k, seed=level)
        total = total[p.cpu().numpy()]
    assert np.array_equal(perm.cpu().numpy(), total)
    ip, ix, _ = ro.permute_csr(indptr, indices, total)
    assert np.array_equal(g_final.indptr.cpu().numpy(), ip)
    assert np.array_equal(g_final.indices.cpu().numpy(), ix)


def test_forty_communities_against_planted_and_grow(ttg_lib):
    import reorder
    rng = np.random.default_rng(7)
    n, k = 40000, 40
    indptr, indices, comm = _community_graph(rng, n, k, 10, 0.9)
    planted = _cut(indptr, indices, comm)
    part, cut = _kway(indptr, indices, k)
    _assert_balanced(part, n, k)
    grow = reorder.grow_partition(_graph(indptr, indices), k).cpu().numpy()
    assert cut <= 1.05 * planted, (cut, planted)
    assert cut < 0.8 * _cut(indptr, indices, grow)


def test_isolated_nodes_and_a_hub_hold_the_bounds(ttg_lib):
    rng = np.random.default_rng(8)
    n, k = 300000, 16
    live = rng.permutation(n)[: int(0.7 * n)]              # 30 % of the nodes stay isolated
    src = rng.choice(live, size=600000)
    dst = rng.choice(live, size=600000)
    hub = int(live[0])
    leaves = rng.choice(live, size=100000, replace=False)
    src = np.concatenate([src, leaves, np.full(100000, hub)])
    dst = np.concatenate([dst, np.full(100000, hub), leaves])
    indptr, indices = _csr(n, src, dst)
    part, cut = _kway(indptr, indices, k)
    _assert_balanced(part, n, k)
    assert cut == _cut(indptr, indices, part)


def test_large_community_graph_recovers_the_planted_partition(ttg_lib):
    import reorder
    import sage
    n, e, k = 1200000, 24000000, 125
    g, comm = sage.synthetic_community_graph(n, e, k, 0.9, DEV, seed=11)
    part, cut = reorder.kway_partition_device(g, k, return_cut=True)
    indptr, indices = g.indptr.cpu().numpy(), g.indices.cpu().numpy()
    planted = _cut(indptr, indices, comm.cpu().numpy())
    p = part.cpu().numpy()
    _assert_balanced(p, n, k)
    assert cut <= 1.02 * planted, (cut, planted)


def test_bad_arguments_are_refused(ttg_lib):
    import _ttg
    import reorder
    indptr, indices = _grid(4, 4)
    g = _graph(indptr, indices)
    with pytest.raises(RuntimeError, match="k=0"):
        reorder.kway_partition_device(g, 0)
    with pytest.raises(RuntimeError, match="k=17"):
        reorder.kway_partition_device(g, 17)
    with pytest.raises(RuntimeError, match="ubfactor"):
        reorder.kway_partition_device(g, 2, ubfactor=0.5)
    bad = indices.copy()
    bad[3] = 16
    with pytest.raises(RuntimeError, match="out of range|outside"):
        reorder.kway_partition_device(_graph(indptr, bad), 2)
    dec = indptr.copy()
    dec[5] = dec[4] - 1                                     # not a CSR: a row ends before it starts
    with pytest.raises(RuntimeError, match="not a CSR"):
        reorder.kway_partition_device(_graph(dec, indices), 2)
    # the C ABI refuses before any CUDA call: k, ubfactor, null pointers, a short workspace
    lib = ttg_lib
    ws = torch.empty(1 << 20, dtype=torch.uint8, device=DEV)
    stream = _ttg.stream_of(torch.device(DEV))
    xa = torch.from_numpy(indptr).to(DEV)
    part = torch.zeros(16, dtype=torch.int32, device=DEV)
    vw = torch.ones(16, dtype=torch.int32, device=DEV)
    stats = (C.c_int64 * 3)()

    def refine(k, ub, pp, nbytes):
        return lib.ttg_kway_refine(16, _ttg.ptr(xa), None, None, _ttg.ptr(vw), 16, k, ub, 1, 0, 0, 0, None, None, pp,
                                   stats, _ttg.ptr(ws), nbytes, stream)
    assert refine(0, 1.03, _ttg.ptr(part), ws.numel()) != 0 and "k=0" in _ttg.last_error()
    assert refine(2, 0.5, _ttg.ptr(part), ws.numel()) != 0 and "ubfactor" in _ttg.last_error()
    assert refine(2, 1.03, None, ws.numel()) != 0 and "null pointer" in _ttg.last_error()
    assert refine(2, 1.03, _ttg.ptr(part), 16) != 0 and "workspace" in _ttg.last_error()
    m = C.c_int64(0)
    assert lib.ttg_kway_symmetrise(16, indices.shape[0], _ttg.ptr(xa), None, None, None, None, None, C.byref(m),
                                   _ttg.ptr(ws), ws.numel(), stream) != 0 and "null pointer" in _ttg.last_error()
