"""Node reordering before training: the role of dgl.reorder_graph in the reference
(graphloader.py:358-372 recursive METIS, :399-454 dgl_partition: 'metis' k / 'rcmk' / random
'custom' permutation), without DGL.

    new_graph, perm = reorder_graph(graph, "rcmk")               # perm[i] = old id of new node i
    new_graph, perm = reorder_graph(graph, "metis", k=125)       # multilevel k-way partition, part by part
    new_graph, perm = recursive_metis_reorder(graph, [50, 60, 60])   # graphloader.py:358-372
    new_graph, perm = reorder_graph(graph, "grow", k=125)        # label propagation on the device
    new_graph, perm = reorder_graph(graph, "custom", nodes_perm=p)
    new_graph, perm = reorder_graph(graph, "degree")             # graphloader.py:275-285: high in-degree first
    labels_new = labels_old[perm]; train_idx_new = inverse(perm)[train_idx_old]

* "rcmk" is exactly what DGL computes: scipy.sparse.csgraph.reverse_cuthill_mckee on the CSR
  adjacency (host, offline preprocessing -- scipy is DGL's own dependency for this).  With
  backend="device" the same permutation, element for element, comes from csrc/rcm.cu
  (ttg_rcm_symmetrise / ttg_rcm_order: symmetrise, components, level-synchronous BFS on the device;
  only numpy.argsort of the degrees runs on the host, because its tie order is part of the result):
      new_graph, perm = reorder_graph(graph, "rcmk", backend="device")
* "metis" is a multilevel k-way partitioner on the host (ttg_partition_kway, csrc/kway_host.cu:
  heavy-edge coarsening, grown initial parts, greedy k-way refinement), where the reference calls
  libmetis through DGL -- host code there too.  Same scheme and balance bound as METIS, not the
  same partition (METIS is not in this image; parity with its order is unpinned).  The new order
  is part by part, old order within a part (stable), as DGL's METIS reorder sorts by part id.
* "grow" partitions on the device (ttg_partition_grow): k connected parts of at most
  ceil(N / k * slack) nodes grown from k seed nodes drawn uniformly (seeded); nodes no part
  could take fill the parts with room.  Much faster than "metis" and a much larger cut.
* the relabelling itself runs on the device (ttg_permute_csr), bit-exact against
  oracle/reorder_oracle.py.
"""
import ctypes as C
import time
from typing import Optional, Tuple

import numpy as np
import torch

import _ttg
from sampler import CSRGraph

_scratch = _ttg._Workspace()


def inverse_permutation(perm: torch.Tensor) -> torch.Tensor:
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(perm.numel(), dtype=perm.dtype, device=perm.device)
    return inv


def permute_graph(g: CSRGraph, perm: torch.Tensor) -> CSRGraph:
    """The graph with new node i = old node perm[i] (in-neighbour lists keep their order)."""
    perm = _ttg.require_cuda(perm, "perm", torch.int64)
    n = g.num_nodes
    if perm.numel() != n:
        raise RuntimeError("permute_graph: perm has %d entries for %d nodes" % (perm.numel(), n))
    dev = perm.device
    lib = _ttg.lib()
    with _ttg.on_device(dev):
        new_indptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
        new_indices = torch.empty(max(g.num_edges, 1), dtype=torch.int32, device=dev)
        inv = torch.empty(n, dtype=torch.int64, device=dev)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        nbytes = lib.ttg_permute_csr_workspace_bytes(n)
        if nbytes == 0:
            raise RuntimeError("permute_graph: %d nodes out of range" % n)
        ws = _scratch.get(dev, nbytes)
        rc = lib.ttg_permute_csr(n, _ttg.ptr(g.indptr), _ttg.ptr(g.indices), _ttg.ptr(perm),
                                 _ttg.ptr(new_indptr), _ttg.ptr(new_indices), _ttg.ptr(inv),
                                 _ttg.ptr(bad), _ttg.ptr(ws), ws.numel(), _ttg.stream_of(dev))
        _ttg.check(rc, "permute_csr")
        # a permutation: every id in range (kernel) and every id hit once (inv o perm = id)
        if int(bad.item()) or not bool((inv[perm] == torch.arange(n, device=dev)).all()):
            raise RuntimeError("permute_graph: perm is not a permutation of 0..%d" % (n - 1))
    return CSRGraph(new_indptr, new_indices[:g.num_edges])


def rcmk_permutation(g: CSRGraph, backend: str = "host", stats: Optional[dict] = None) -> torch.Tensor:
    """reverse Cuthill-McKee order, computed the way DGL's 'rcmk' does: scipy on the host
    (backend="host") or csrc/rcm.cu (backend="device", the same permutation).  With the device
    backend `stats`, when given, receives the seconds of each phase and the numbers of BFS levels
    and connected components."""
    if backend == "device":
        return _rcmk_device(g, stats)
    if backend != "host":
        raise RuntimeError("rcmk_permutation: unknown backend %r (host or device)" % backend)
    from scipy import sparse
    n = g.num_nodes
    indptr = g.indptr.cpu().numpy()
    indices = g.indices.cpu().numpy()
    adj = sparse.csr_matrix((np.ones(indices.shape[0], dtype=np.int8), indices, indptr), shape=(n, n))
    perm = sparse.csgraph.reverse_cuthill_mckee(adj, symmetric_mode=False)
    return torch.from_numpy(np.ascontiguousarray(perm).astype(np.int64)).to(g.indptr.device)


def _rcmk_device(g: CSRGraph, stats: Optional[dict]) -> torch.Tensor:
    n, dev = g.num_nodes, g.indptr.device
    if n == 0:
        return torch.empty(0, dtype=torch.int64, device=dev)
    lib = _ttg.lib()
    with _ttg.on_device(dev):
        t0 = time.perf_counter()
        nnz = int(g.indptr[-1])
        if nnz > g.num_edges:
            raise RuntimeError("rcmk_permutation: indptr[-1] = %d > %d indices" % (nnz, g.num_edges))
        sym_indptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
        sym_indices = torch.empty(max(2 * nnz, 1), dtype=torch.int32, device=dev)
        degree = torch.empty(n, dtype=torch.int32, device=dev)
        sym_edges = C.c_int64(0)
        nbytes = lib.ttg_rcm_symmetrise_workspace_bytes(n, nnz)
        if nbytes == 0:
            raise RuntimeError("rcmk_permutation: %d nodes / %d edges out of range" % (n, nnz))
        # ~24 bytes per symmetrised entry (7 GB at products shape): a buffer of this call alone, not the
        # module's scratch that lives as long as the process
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        rc = lib.ttg_rcm_symmetrise(n, nnz, _ttg.ptr(g.indptr), _ttg.ptr(g.indices), _ttg.ptr(sym_indptr),
                                    _ttg.ptr(sym_indices), _ttg.ptr(degree), C.byref(sym_edges), _ttg.ptr(ws),
                                    ws.numel(), _ttg.stream_of(dev))
        _ttg.check(rc, "rcm_symmetrise")
        del ws
        torch.cuda.current_stream(dev).synchronize()
        t1 = time.perf_counter()
        # scipy's own call, on the host: numpy's tie order among equal degrees is part of the result
        rank_nodes = torch.from_numpy(np.argsort(degree.cpu().numpy())).to(dev)
        t2 = time.perf_counter()
        perm = torch.empty(n, dtype=torch.int64, device=dev)
        counts = (C.c_int64 * 2)()
        phase_ms = (C.c_double * 3)()
        ws = torch.empty(lib.ttg_rcm_order_workspace_bytes(n), dtype=torch.uint8, device=dev)
        rc = lib.ttg_rcm_order(n, sym_edges.value, _ttg.ptr(sym_indptr), _ttg.ptr(sym_indices), _ttg.ptr(degree),
                               _ttg.ptr(rank_nodes), _ttg.ptr(perm), counts, phase_ms, _ttg.ptr(ws), ws.numel(),
                               _ttg.stream_of(dev))
        _ttg.check(rc, "rcm_order")
    del ws
    if stats is not None:
        stats.update(symmetrise_s=t1 - t0, host_argsort_s=t2 - t1, components_s=phase_ms[0] / 1e3,
                     bfs_s=phase_ms[1] / 1e3, order_s=phase_ms[2] / 1e3, levels=int(counts[0]),
                     components=int(counts[1]), sym_edges=int(sym_edges.value))
    return perm


def grow_partition(g: CSRGraph, k: int, slack: float = 1.03, seed: int = 0,
                   sweeps_per_call: int = 8, max_calls: int = 64) -> torch.Tensor:
    """int32 part id of every node: k parts of at most ceil(N / k * slack) nodes."""
    n, dev = g.num_nodes, g.indptr.device
    k = int(k)
    if not 0 < k <= n:
        raise RuntimeError("grow_partition: k=%d out of range" % k)
    cap = int(np.ceil(n / k * slack))
    gen = torch.Generator(device="cpu").manual_seed(seed)
    seeds = torch.randperm(n, generator=gen)[:k].to(dev)
    lib = _ttg.lib()
    with _ttg.on_device(dev):
        la = torch.empty(n, dtype=torch.int32, device=dev)
        lb = torch.empty(n, dtype=torch.int32, device=dev)
        sizes = torch.empty(k, dtype=torch.int32, device=dev)
        changed = torch.zeros(1, dtype=torch.int32, device=dev)
        for call in range(max_calls):
            rc = lib.ttg_partition_grow(n, _ttg.ptr(g.indptr), _ttg.ptr(g.indices), k, cap,
                                        _ttg.ptr(seeds) if call == 0 else None, sweeps_per_call,
                                        _ttg.ptr(la), _ttg.ptr(lb), _ttg.ptr(sizes), _ttg.ptr(changed),
                                        _ttg.stream_of(dev))
            _ttg.check(rc, "partition_grow")
            if int(changed.item()) == 0:
                break
        # leftovers (isolated nodes, or every neighbouring part full): fill the parts with room
        left = torch.nonzero(la < 0).flatten()
        if left.numel():
            room = (cap - sizes.long()).clamp_min(0)
            slots = torch.repeat_interleave(torch.arange(k, device=dev), room)
            la[left] = slots[:left.numel()].int()
    return la


def kway_partition(g: CSRGraph, k: int, ubfactor: float = 1.03, seed: int = 0, refine_passes: int = 10,
                   return_cut: bool = False):
    """int32 part id of every node from the multilevel k-way partitioner (host code, like the METIS
    call it stands for: dgl.metis_partition_assignment behind graphloader.py:370,440); parts hold at
    most ubfactor * ceil(N / k) nodes.  The graph is copied to the host and the labels come back
    on the graph's device.  With return_cut also the number of edges between different parts."""
    n, dev = g.num_nodes, g.indptr.device
    k = int(k)
    if not 0 < k <= max(n, 1):
        raise RuntimeError("kway_partition: k=%d out of range" % k)
    indptr = np.ascontiguousarray(g.indptr.cpu().numpy(), dtype=np.int64)
    indices = np.ascontiguousarray(g.indices.cpu().numpy()[:int(indptr[-1])], dtype=np.int32)
    part = np.empty(n, dtype=np.int32)
    cut = C.c_int64(0)
    rc = _ttg.lib().ttg_partition_kway(n, indptr.ctypes.data, indices.ctypes.data, k, float(ubfactor), int(seed),
                                       int(refine_passes), part.ctypes.data, C.byref(cut))
    _ttg.check(rc, "partition_kway")
    labels = torch.from_numpy(part).to(dev)
    return (labels, int(cut.value)) if return_cut else labels


def degree_permutation(g: CSRGraph, percentile: float = 80.0) -> torch.Tensor:
    """graphloader.py:275-285 (custom_reordering, is_degree=True): the nodes whose in-degree reaches the
    `percentile`-th percentile of all in-degrees first, the others behind them, both in increasing id."""
    deg = (g.indptr[1:] - g.indptr[:-1]).to(torch.float64)
    if deg.numel() == 0:
        return torch.empty(0, dtype=torch.int64, device=g.indptr.device)
    # np.percentile's default (linear interpolation between the two nearest ranks), on the host in fp64:
    # torch.quantile refuses more than 16 M elements
    threshold = float(np.percentile(deg.cpu().numpy(), percentile))
    high = deg >= threshold
    ids = torch.arange(deg.numel(), dtype=torch.int64, device=deg.device)
    return torch.cat([ids[high], ids[~high]])


def partition_permutation(labels: torch.Tensor) -> torch.Tensor:
    """Part by part, old order inside a part (stable sort by part id)."""
    return torch.sort(labels.long(), stable=True).indices


def reorder_graph(g: CSRGraph, algo: str, k: Optional[int] = None,
                  nodes_perm: Optional[torch.Tensor] = None, seed: int = 0, backend: str = "host"
                  ) -> Tuple[CSRGraph, torch.Tensor]:
    """backend selects where "rcmk" runs ("host": scipy, "device": csrc/rcm.cu, the same order); the
    other algorithms have one implementation each and refuse backend="device"."""
    if backend not in ("host", "device"):
        raise RuntimeError("reorder_graph: unknown backend %r (host or device)" % backend)
    if backend != "host" and algo != "rcmk":
        raise RuntimeError("reorder_graph: backend=%r applies to 'rcmk' only, not %r" % (backend, algo))
    if algo == "custom":
        if nodes_perm is None:
            raise RuntimeError("reorder_graph('custom') needs nodes_perm")
        perm = nodes_perm.to(g.indptr.device, torch.int64).contiguous()
    elif algo == "rcmk":
        perm = rcmk_permutation(g, backend)
    elif algo == "degree":
        perm = degree_permutation(g)
    elif algo == "grow":
        if k is None:
            raise RuntimeError("reorder_graph('grow') needs k")
        perm = partition_permutation(grow_partition(g, k, seed=seed))
    elif algo == "metis":
        if k is None:
            raise RuntimeError("reorder_graph('metis') needs k")
        perm = partition_permutation(kway_partition(g, k, seed=seed))
    else:
        raise RuntimeError("reorder_graph: unknown algorithm %r" % algo)
    return permute_graph(g, perm), perm


def recursive_metis_reorder(g: CSRGraph, partition_list, seed: int = 0) -> Tuple[CSRGraph, torch.Tensor]:
    """graphloader.py:358-372: one 'metis' reorder per entry of partition_list ([50, 60, 60] at
    :432), each applied to the graph the previous one produced.  Returns the final graph and the
    composed permutation (perm[i] = id in the ORIGINAL graph of final node i)."""
    perm = torch.arange(g.num_nodes, dtype=torch.int64, device=g.indptr.device)
    for level, k in enumerate(partition_list):
        g, p = reorder_graph(g, "metis", k=int(k), seed=seed + level)
        perm = perm[p]
    return g, perm
