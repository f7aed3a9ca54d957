"""Node reordering on the GPU (csrc/reorder.cu, reorder.py) against oracle/reorder_oracle.py."""
import numpy as np
import pytest
import torch

from oracle import reorder_oracle as ro

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _community_graph(rng, n, k, deg, p_in):
    """k equal communities with scrambled ids; symmetric edges."""
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


def _to_graph(indptr, indices):
    from sampler import CSRGraph
    return CSRGraph(torch.from_numpy(indptr).to(DEV), torch.from_numpy(indices).to(DEV))


@pytest.mark.parametrize("n,e", [(1, 0), (5, 3), (1000, 20000), (4097, 100)])
def test_permute_graph_is_bit_exact(ttg_lib, n, e):
    import reorder
    rng = np.random.default_rng(n)
    deg = rng.multinomial(e, np.ones(n) / n)
    indptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int64)
    indices = rng.integers(0, n, size=e).astype(np.int32)
    perm = rng.permutation(n).astype(np.int64)
    g2 = reorder.permute_graph(_to_graph(indptr, indices), torch.from_numpy(perm).to(DEV))
    ip, ix, _ = ro.permute_csr(indptr, indices, perm)
    assert np.array_equal(g2.indptr.cpu().numpy(), ip)
    assert np.array_equal(g2.indices.cpu().numpy(), ix)


def test_permute_graph_rejects_non_permutations(ttg_lib):
    import reorder
    g = _to_graph(np.array([0, 1, 2, 3], dtype=np.int64), np.array([1, 2, 0], dtype=np.int32))
    for bad in ([0, 1, 3], [0, 0, 1], [0, 1]):
        with pytest.raises(RuntimeError):
            reorder.permute_graph(g, torch.tensor(bad, dtype=torch.int64, device=DEV))


@pytest.mark.parametrize("fault", ["id_equal_to_n", "negative_id", "decreasing_indptr", "indptr0_not_zero",
                                   "indptr_beyond_indices"])
def test_permute_graph_refuses_a_bad_graph(ttg_lib, fault):
    """Under a valid permutation the graph itself is checked, before any id is looked up or any row is copied."""
    import reorder
    indptr = np.array([0, 2, 3, 5], dtype=np.int64)
    indices = np.array([1, 2, 0, 0, 1], dtype=np.int32)
    if fault == "id_equal_to_n":
        indices[2] = 3
    elif fault == "negative_id":
        indices[4] = -1
    elif fault == "decreasing_indptr":
        indptr[1] = 4
    elif fault == "indptr0_not_zero":
        indptr[0] = 1
    else:
        indptr[3] = 6
    with pytest.raises(RuntimeError, match=r"graph is not a CSR|indptr\[-1\] = 6 > 5 indices"):
        reorder.permute_graph(_to_graph(indptr, indices), torch.tensor([2, 0, 1], dtype=torch.int64, device=DEV))


def test_rcmk_is_scipys_order_and_reduces_bandwidth(ttg_lib):
    import reorder
    from scipy import sparse
    # a band graph (i ~ i +- 1, i +- 2) under scrambled ids: RCM finds the band again
    rng = np.random.default_rng(3)
    n = 3000
    scr = rng.permutation(n)
    a = np.arange(n)
    pairs = np.concatenate([np.stack([a[:-1], a[1:]], 1), np.stack([a[:-2], a[2:]], 1)])
    src = scr[np.concatenate([pairs[:, 0], pairs[:, 1]])]
    dst = scr[np.concatenate([pairs[:, 1], pairs[:, 0]])]
    order = np.lexsort((src, dst))
    src, dst = src[order], dst[order]
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(dst, minlength=n), out=indptr[1:])
    indices = src.astype(np.int32)
    g = _to_graph(indptr, indices)
    g2, perm = reorder.reorder_graph(g, "rcmk")
    adj = sparse.csr_matrix((np.ones(indices.shape[0], dtype=np.int8), indices, indptr), shape=(n, n))
    assert np.array_equal(perm.cpu().numpy(), sparse.csgraph.reverse_cuthill_mckee(adj, symmetric_mode=False))

    def bandwidth(ip, ix):
        d = np.repeat(np.arange(ip.shape[0] - 1), np.diff(ip))
        return np.abs(d - ix).max()
    assert bandwidth(indptr, indices) > 1000
    assert bandwidth(g2.indptr.cpu().numpy(), g2.indices.cpu().numpy()) <= 4


def test_grow_partition_invariants_and_locality(ttg_lib):
    import reorder
    rng = np.random.default_rng(4)
    n, k = 20000, 40
    indptr, indices, comm = _community_graph(rng, n, k, 8, 0.9)
    g = _to_graph(indptr, indices)
    labels = reorder.grow_partition(g, k, slack=1.05, seed=1)
    lab = labels.cpu().numpy()
    assert lab.min() >= 0 and lab.max() < k
    assert np.bincount(lab, minlength=k).max() <= int(np.ceil(n / k * 1.05))
    g2, perm = reorder.reorder_graph(g, "grow", k=k, seed=1)
    p = perm.cpu().numpy()
    assert np.array_equal(np.sort(p), np.arange(n))
    # the reordered graph is the oracle's relabelling under that permutation
    ip, ix, _ = ro.permute_csr(indptr, indices, p)
    assert np.array_equal(g2.indptr.cpu().numpy(), ip) and np.array_equal(g2.indices.cpu().numpy(), ix)
    # locality: far more edges stay inside a block of n / k consecutive ids than before
    def inside(ip_, ix_):
        dst = np.repeat(np.arange(n), np.diff(ip_))
        return np.mean(dst // (n // k) == ix_ // (n // k))
    assert inside(ip, ix) > 5 * inside(indptr, indices)


def test_metis_reorder_is_part_by_part_and_local(ttg_lib):
    """reorder_graph(g, 'metis', k) (graphloader.py:440): the multilevel k-way partition of
    csrc/kway_host.cu, nodes sorted by part (stable), relabelled on the device."""
    import reorder
    rng = np.random.default_rng(5)
    n, k = 20000, 40
    indptr, indices, comm = _community_graph(rng, n, k, 8, 0.9)
    g = _to_graph(indptr, indices)
    labels, cut = reorder.kway_partition(g, k, seed=1, return_cut=True)
    lab = labels.cpu().numpy()
    assert labels.device.type == "cuda" and lab.min() == 0 and lab.max() == k - 1
    assert np.bincount(lab, minlength=k).max() <= int(1.03 * np.ceil(n / k))
    dst = np.repeat(np.arange(n), np.diff(indptr))
    assert cut == int((lab[dst] != lab[indices]).sum())
    assert cut <= 1.05 * int((comm[dst] != comm[indices]).sum())       # the planted communities, or better
    g2, perm = reorder.reorder_graph(g, "metis", k=k, seed=1)
    p = perm.cpu().numpy()
    assert np.array_equal(np.sort(p), np.arange(n))
    assert np.all(np.diff(lab[p]) >= 0)                               # part by part ...
    for c in (0, k // 2, k - 1):                                      # ... old order inside a part
        assert np.all(np.diff(p[lab[p] == c]) > 0)
    ip, ix, _ = ro.permute_csr(indptr, indices, p)
    assert np.array_equal(g2.indptr.cpu().numpy(), ip) and np.array_equal(g2.indices.cpu().numpy(), ix)
    # far fewer edges leave a part than the device-side label propagation leaves ("grow")
    grow = reorder.grow_partition(g, k, slack=1.05, seed=1).cpu().numpy()
    assert cut < 0.8 * int((grow[dst] != grow[indices]).sum())


def test_recursive_metis_reorder_composes_the_permutations(ttg_lib):
    """graphloader.py:358-372: one METIS reorder per level on the graph the previous level left."""
    import reorder
    rng = np.random.default_rng(6)
    n = 6000
    indptr, indices, _ = _community_graph(rng, n, 12, 6, 0.85)
    g = _to_graph(indptr, indices)
    g3, perm = reorder.recursive_metis_reorder(g, [4, 6, 12])
    p = perm.cpu().numpy()
    assert np.array_equal(np.sort(p), np.arange(n))
    ip, ix, _ = ro.permute_csr(indptr, indices, p)
    assert np.array_equal(g3.indptr.cpu().numpy(), ip) and np.array_equal(g3.indices.cpu().numpy(), ix)


def test_unknown_algorithms_fail_loudly(ttg_lib):
    import reorder
    g = _to_graph(np.array([0, 1, 2], dtype=np.int64), np.array([1, 0], dtype=np.int32))
    with pytest.raises(RuntimeError):
        reorder.reorder_graph(g, "nope", k=2)
    with pytest.raises(RuntimeError):
        reorder.reorder_graph(g, "metis")          # k is required


def test_degree_reorder_is_the_reference_expression(ttg_lib):
    """graphloader.py:275-285 restated with numpy: nodes at or above the 80th percentile of the in-degrees first."""
    import reorder
    rng = np.random.default_rng(8)
    n, e = 5000, 60000
    deg = rng.multinomial(e, rng.dirichlet(np.full(n, 0.3)))
    indptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int64)
    indices = rng.integers(0, n, size=e).astype(np.int32)
    g = _to_graph(indptr, indices)
    degrees = np.diff(indptr)
    high = np.where(degrees >= np.percentile(degrees, 80))[0]
    want = np.concatenate((high, np.setdiff1d(np.arange(n), high)))
    g2, perm = reorder.reorder_graph(g, "degree")
    assert np.array_equal(perm.cpu().numpy(), want)
    ip, ix, _ = ro.permute_csr(indptr, indices, want)
    assert np.array_equal(g2.indptr.cpu().numpy(), ip) and np.array_equal(g2.indices.cpu().numpy(), ix)
