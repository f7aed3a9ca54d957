"""Reverse Cuthill-McKee on the device (csrc/rcm.cu, reorder_graph(g, "rcmk", backend="device")):
the same permutation as scipy's, element for element, and the same relabelled graph."""
import numpy as np
import pytest
import torch

from oracle import rcm_oracle as ro
from oracle import reorder_oracle as rorc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _to_graph(indptr, indices):
    from sampler import CSRGraph
    return CSRGraph(torch.from_numpy(indptr).to(DEV), torch.from_numpy(indices).to(DEV))


def _same_as_scipy(g, stats=None):
    """Device path against the scipy path: permutation and relabelled CSR; returns the permutation."""
    import reorder
    g_host, p_host = reorder.reorder_graph(g, "rcmk")
    g_dev, p_dev = reorder.reorder_graph(g, "rcmk", backend="device")
    want = p_host.cpu().numpy()
    got = p_dev.cpu().numpy()
    assert p_dev.dtype == torch.int64 and p_dev.device == g.indptr.device
    assert np.array_equal(got, want), "first difference at %d" % int(np.argmax(got != want))
    assert torch.equal(g_dev.indptr, g_host.indptr) and torch.equal(g_dev.indices, g_host.indices)
    if stats is not None:
        reorder.rcmk_permutation(g, backend="device", stats=stats)
    return got


def test_every_family_matches_scipy(ttg_lib):
    rng = np.random.default_rng(77)
    for t in range(400):
        kind, indptr, indices = ro.random_case(rng, t)
        g = _to_graph(indptr, indices)
        stats = {}
        _same_as_scipy(g, stats)
        perm, (levels, comps) = ro.rcm_order(indptr, indices, return_stats=True)
        assert (stats["levels"], stats["components"]) == (levels, comps), (t, kind)
        ptr, _ = ro.sym_lists(indptr, indices)
        assert stats["sym_edges"] == int(ptr[-1])


def test_scrambled_band_graph(ttg_lib):
    """The band graph of test_gpu_reorder.py (i ~ i +- 1, i +- 2 under scrambled ids)."""
    rng = np.random.default_rng(3)
    n = 3000
    scr = rng.permutation(n)
    a = np.arange(n)
    pairs = np.concatenate([np.stack([a[:-1], a[1:]], 1), np.stack([a[:-2], a[2:]], 1)])
    src = scr[np.concatenate([pairs[:, 0], pairs[:, 1]])]
    dst = scr[np.concatenate([pairs[:, 1], pairs[:, 0]])]
    indptr, indices = ro.csr_from_edges(n, src, dst, canonical=True)
    _same_as_scipy(_to_graph(indptr, indices))


def test_long_path_has_one_level_per_node(ttg_lib):
    rng = np.random.default_rng(5)
    n = 20000
    scr = rng.permutation(n)
    src = scr[np.concatenate([np.arange(n - 1), np.arange(1, n)])]
    dst = scr[np.concatenate([np.arange(1, n), np.arange(n - 1)])]
    indptr, indices = ro.csr_from_edges(n, src, dst, canonical=False)
    stats = {}
    _same_as_scipy(_to_graph(indptr, indices), stats)
    assert stats["components"] == 1 and stats["levels"] == n


def test_star(ttg_lib):
    n = 5001
    leaves = np.arange(1, n)
    for canonical in (True, False):
        src = np.concatenate([leaves, np.zeros(n - 1, np.int64)])
        dst = np.concatenate([np.zeros(n - 1, np.int64), leaves])
        indptr, indices = ro.csr_from_edges(n, src, dst, canonical)
        stats = {}
        _same_as_scipy(_to_graph(indptr, indices), stats)
        assert stats["levels"] == 3 and stats["components"] == 1


def test_thousands_of_components(ttg_lib):
    rng = np.random.default_rng(9)
    sizes = rng.integers(1, 12, 2500)
    n = int(sizes.sum())
    base = np.repeat(np.concatenate([[0], np.cumsum(sizes)[:-1]]), 3 * sizes)
    span = np.repeat(sizes, 3 * sizes)
    src = base + (rng.random(base.shape[0]) * span).astype(np.int64)
    dst = base + (rng.random(base.shape[0]) * span).astype(np.int64)
    scr = rng.permutation(n)
    indptr, indices = ro.csr_from_edges(n, scr[src], scr[dst], canonical=False)
    stats = {}
    _same_as_scipy(_to_graph(indptr, indices), stats)
    assert stats["components"] > 1000


def test_community_graph(ttg_lib):
    import sage
    g, _ = sage.synthetic_community_graph(50000, 600000, 25, 0.9, torch.device(DEV), seed=1)
    _same_as_scipy(g)


def test_large_power_law_graph_and_repeatability(ttg_lib):
    import reorder
    import sage
    g = sage.synthetic_graph(400000, 10_500_000, torch.device(DEV), seed=3)
    assert g.num_edges >= 10_000_000
    first = _same_as_scipy(g)
    again = reorder.rcmk_permutation(g, backend="device")
    assert np.array_equal(again.cpu().numpy(), first)


def test_backend_refused_for_other_algorithms(ttg_lib):
    import reorder
    g = _to_graph(np.array([0, 1, 2], np.int64), np.array([1, 0], np.int32))
    for algo, kw in (("metis", {"k": 2}), ("grow", {"k": 2}), ("degree", {}),
                     ("custom", {"nodes_perm": torch.tensor([1, 0])})):
        with pytest.raises(RuntimeError, match="backend"):
            reorder.reorder_graph(g, algo, backend="device", **kw)
    with pytest.raises(RuntimeError, match="backend"):
        reorder.reorder_graph(g, "rcmk", backend="scipy")


def test_bad_ids_are_refused(ttg_lib):
    import reorder
    g = _to_graph(np.array([0, 1, 2], np.int64), np.array([1, 7], np.int32))
    with pytest.raises(RuntimeError, match="outside"):
        reorder.rcmk_permutation(g, backend="device")
    g = _to_graph(np.array([1, 2, 3], np.int64), np.array([1, 0, 1], np.int32))   # indptr[0] != 0
    with pytest.raises(RuntimeError, match="indptr"):
        reorder.rcmk_permutation(g, backend="device")
