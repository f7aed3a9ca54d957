"""Node reordering before training: the role of dgl.reorder_graph in the reference
(graphloader.py:358-372 recursive METIS, :399-454 dgl_partition: 'metis' k / 'rcmk' / random
'custom' permutation), without DGL.

    new_graph, perm = reorder_graph(graph, "rcmk")               # perm[i] = old id of new node i
    new_graph, perm = reorder_graph(graph, "metis", k=125)       # multilevel k-way partition, part by part
    new_graph, perm = recursive_metis_reorder(graph, [50, 60, 60])   # graphloader.py:358-372
    new_graph, perm = reorder_graph(graph, "kway", k=125)        # multilevel k-way on the device
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
* "kway" is the same multilevel scheme with its data-parallel steps on the device
  (kway_partition_device, csrc/kway.cu: sort-based symmetrise, handshake heavy-edge matching and
  contraction level by level, the host partitioner's grown initial parts on the coarsest graph,
  Jet-style synchronous label propagation with an afterburner and sorted admission on the way up).
  The same balance bounds and cut quality bar as "metis", a different partition (neither the host
  partitioner's nor METIS'); device-only, so it takes no backend:
      new_graph, perm = reorder_graph(graph, "kway", k=125)
      new_graph, perm = recursive_metis_reorder(graph, [50, 60, 60], algo="kway")
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


def _edge_count(g: CSRGraph, who: str) -> int:
    """indptr[-1], the entries the in-lists use; refused when the indices array holds fewer"""
    nnz = int(g.indptr[-1])
    if nnz > g.num_edges:
        raise RuntimeError("%s: indptr[-1] = %d > %d indices" % (who, nnz, g.num_edges))
    return nnz


def _workspace(dev, who: str, query, **sizes) -> torch.Tensor:
    """A workspace of one call alone: the symmetrise ones take ~24 bytes per symmetrised entry (7 GB at products
    shape), too much to keep for the process.  A size of 0 is the C side refusing `sizes` (in query order)."""
    nbytes = query(*sizes.values())
    if nbytes == 0:
        raise RuntimeError("%s: %s out of range" % (who, " / ".join("%d %s" % (v, k) for k, v in sizes.items())))
    return torch.empty(nbytes, dtype=torch.uint8, device=dev)


def _check_k(who: str, k: int, n: int, ubfactor: float) -> int:
    k = int(k)
    if not 0 < k <= max(n, 1):
        raise RuntimeError("%s: k=%d out of range" % (who, k))
    if ubfactor < 1.0:
        raise RuntimeError("%s: ubfactor %g below 1" % (who, ubfactor))
    return k


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
        _edge_count(g, "permute_graph")
        new_indptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
        new_indices = torch.empty(max(g.num_edges, 1), dtype=torch.int32, device=dev)
        inv = torch.empty(n, dtype=torch.int64, device=dev)
        bad = torch.zeros(1, dtype=torch.int32, device=dev)
        ws = _workspace(dev, "permute_graph", lib.ttg_permute_csr_workspace_bytes, nodes=n)
        rc = lib.ttg_permute_csr(n, _ttg.ptr(g.indptr), _ttg.ptr(g.indices), _ttg.ptr(perm),
                                 _ttg.ptr(new_indptr), _ttg.ptr(new_indices), _ttg.ptr(inv),
                                 _ttg.ptr(bad), _ttg.ptr(ws), ws.numel(), _ttg.stream_of(dev))
        _ttg.check(rc, "permute_csr")
        flags = int(bad.item())   # bit 0: a perm id out of range, bit 1: a bad row or in-neighbour id
        if flags == 2:
            raise RuntimeError("permute_graph: the graph is not a CSR of %d nodes with ids in [0, %d)" % (n, n))
        # a permutation: every id in range (kernel) and every id hit once (inv o perm = id)
        if flags or not bool((inv[perm] == torch.arange(n, device=dev)).all()):
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
        nnz = _edge_count(g, "rcmk_permutation")
        sym_indptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
        sym_indices = torch.empty(max(2 * nnz, 1), dtype=torch.int32, device=dev)
        degree = torch.empty(n, dtype=torch.int32, device=dev)
        sym_edges = C.c_int64(0)
        ws = _workspace(dev, "rcmk_permutation", lib.ttg_rcm_symmetrise_workspace_bytes, nodes=n, edges=nnz)
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
        ws = _workspace(dev, "rcmk_permutation", lib.ttg_rcm_order_workspace_bytes, nodes=n)
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
    k = _check_k("kway_partition", k, n, ubfactor)
    indptr = np.ascontiguousarray(g.indptr.cpu().numpy(), dtype=np.int64)
    indices = np.ascontiguousarray(g.indices.cpu().numpy()[:int(indptr[-1])], dtype=np.int32)
    part = np.empty(n, dtype=np.int32)
    cut = C.c_int64(0)
    rc = _ttg.lib().ttg_partition_kway(n, indptr.ctypes.data, indices.ctypes.data, k, float(ubfactor), int(seed),
                                       int(refine_passes), part.ctypes.data, C.byref(cut))
    _ttg.check(rc, "partition_kway")
    labels = torch.from_numpy(part).to(dev)
    return (labels, int(cut.value)) if return_cut else labels


def kway_partition_device(g: CSRGraph, k: int, ubfactor: float = 1.03, seed: int = 0, refine_passes: int = 10,
                          return_cut: bool = False, stats: Optional[dict] = None):
    """int32 part id of every node from the multilevel k-way partitioner on the device (csrc/kway.cu); the
    contract of kway_partition: every part holds at most max(ceil(N / k), ubfactor * ceil(N / k)) nodes and at
    least floor(N / k) / ubfactor, the labels are on the graph's device and depend on the graph and the seed
    alone; with return_cut also the number of input edges whose ends lie in different parts.  The partition
    is not kway_partition's (nor METIS'): the matching and the refinement are parallel formulations.  Only the
    initial parts of the coarsest graph are computed on the host, by the host partitioner's own code.  `stats`,
    when given, receives the seconds of each phase, the number of levels and the coarsest graph's size."""
    n, dev = g.num_nodes, g.indptr.device
    k = _check_k("kway_partition_device", k, n, ubfactor)
    if n == 0 or k == 1:
        labels = torch.zeros(n, dtype=torch.int32, device=dev)
        return (labels, 0) if return_cut else labels
    lib = _ttg.lib()
    stream = _ttg.stream_of(dev)
    ub = float(ubfactor)
    times = {}
    with _ttg.on_device(dev):
        sync = torch.cuda.current_stream(dev).synchronize
        t0 = time.perf_counter()
        nnz = _edge_count(g, "kway_partition_device")
        xadj = torch.empty(n + 1, dtype=torch.int64, device=dev)
        adj = torch.empty(max(2 * nnz, 1), dtype=torch.int32, device=dev)
        adjw = torch.empty(max(2 * nnz, 1), dtype=torch.int32, device=dev)
        vw = torch.empty(n, dtype=torch.int32, device=dev)
        m = C.c_int64(0)
        ws = _workspace(dev, "kway_partition_device", lib.ttg_kway_symmetrise_workspace_bytes, nodes=n, edges=nnz)
        _ttg.check(lib.ttg_kway_symmetrise(n, nnz, _ttg.ptr(g.indptr), _ttg.ptr(g.indices), _ttg.ptr(xadj),
                                           _ttg.ptr(adj), _ttg.ptr(adjw), _ttg.ptr(vw), C.byref(m), _ttg.ptr(ws),
                                           ws.numel(), stream), "kway_symmetrise")
        del ws
        # trim the symmetrised lists to their size: every level is kept for the way back up
        levels = [(n, m.value, xadj, adj[:m.value].clone(), adjw[:m.value].clone(), vw)]
        del adj, adjw
        t1 = time.perf_counter()
        times["symmetrise_s"] = t1 - t0
        # the host partitioner's stopping rules and vertex-weight bound
        cmaps = []
        coarsen_to = max(30 * k, 256)
        maxvw = max(1, 3 * n // (2 * coarsen_to))
        counts = (C.c_int64 * 2)()
        while levels[-1][0] > coarsen_to and len(levels) < 48:
            ln, lm, lx, la, lw, lv = levels[-1]
            cmap = torch.empty(ln, dtype=torch.int32, device=dev)
            cx = torch.empty(ln + 1, dtype=torch.int64, device=dev)
            ca = torch.empty(max(lm, 1), dtype=torch.int32, device=dev)
            cw = torch.empty(max(lm, 1), dtype=torch.int32, device=dev)
            cv = torch.empty(ln, dtype=torch.int32, device=dev)
            ws = _workspace(dev, "kway_partition_device", lib.ttg_kway_coarsen_workspace_bytes, nodes=ln, edges=lm)
            _ttg.check(lib.ttg_kway_coarsen(ln, lm, _ttg.ptr(lx), _ttg.ptr(la), _ttg.ptr(lw), _ttg.ptr(lv), maxvw,
                                            int(seed), len(levels) - 1, _ttg.ptr(cmap), _ttg.ptr(cx), _ttg.ptr(ca),
                                            _ttg.ptr(cw), _ttg.ptr(cv), counts, _ttg.ptr(ws), ws.numel(), stream),
                       "kway_coarsen")
            del ws
            cn, cm = int(counts[0]), int(counts[1])
            if cn > ln - ln // 20:   # the matching stalls (< 5 % fewer vertices)
                break
            cmaps.append(cmap)
            levels.append((cn, cm, cx[:cn + 1].clone(), ca[:cm].clone(), cw[:cm].clone(), cv[:cn].clone()))
        t2 = time.perf_counter()
        times["coarsen_s"] = t2 - t1
        # initial parts on the host: the host partitioner's grown trials and their refinement
        cn, cm, cx, ca, cw, cv = levels[-1]
        hx, ha, hw, hv = (np.ascontiguousarray(t.cpu().numpy()) for t in (cx, ca, cw, cv))
        hpart = np.empty(cn, dtype=np.int32)
        _ttg.check(lib.ttg_partition_kway_initial(cn, hx.ctypes.data, ha.ctypes.data if cm else None,
                                                  hw.ctypes.data if cm else None, hv.ctypes.data, n, k, ub,
                                                  int(seed), int(refine_passes), hpart.ctypes.data),
                   "partition_kway_initial")
        part = torch.from_numpy(hpart).to(dev)
        t3 = time.perf_counter()
        times["host_initial_s"] = t3 - t2
        rstats = (C.c_int64 * 3)()
        iterations = fills = 0
        for lv in range(len(levels) - 1, -1, -1):
            ln, lm, lx, la, lw, lvw = levels[lv]
            if lv < len(levels) - 1:
                fine = torch.empty(ln, dtype=torch.int32, device=dev)
                cmap, coarse = cmaps[lv], part
            else:
                fine, cmap, coarse = part, None, None
            ws = _workspace(dev, "kway_partition_device", lib.ttg_kway_refine_workspace_bytes, nodes=ln, parts=k)
            _ttg.check(lib.ttg_kway_refine(ln, _ttg.ptr(lx), _ttg.ptr(la) if lm else None,
                                           _ttg.ptr(lw) if lm else None, _ttg.ptr(lvw), n, k, ub, int(lv == 0),
                                           int(seed), lv, int(refine_passes), _ttg.ptr(cmap), _ttg.ptr(coarse),
                                           _ttg.ptr(fine), rstats, _ttg.ptr(ws), ws.numel(), stream), "kway_refine")
            del ws
            part = fine
            iterations += int(rstats[0])
            fills += int(rstats[2])
            levels[lv] = None   # this level's graph is done with
        sync()
        t4 = time.perf_counter()
        times["refine_s"] = t4 - t3
        cut = C.c_int64(0)
        if (return_cut or stats is not None) and nnz > 0:
            ws = _workspace(dev, "kway_partition_device", lib.ttg_kway_edge_cut_workspace_bytes)
            _ttg.check(lib.ttg_kway_edge_cut(n, _ttg.ptr(g.indptr), _ttg.ptr(g.indices), _ttg.ptr(part),
                                             C.byref(cut), _ttg.ptr(ws), ws.numel(), stream), "kway_edge_cut")
    if stats is not None:
        stats.update(times, levels=len(cmaps) + 1, coarsest_nodes=cn, coarsest_edges=cm, sym_edges=m.value,
                     refine_iterations=iterations, exact_fills=fills, cut=int(cut.value))
    return (part, int(cut.value)) if return_cut else part


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
    if algo in ("grow", "metis", "kway") and k is None:
        raise RuntimeError("reorder_graph(%r) needs k" % algo)
    if algo == "custom":
        if nodes_perm is None:
            raise RuntimeError("reorder_graph('custom') needs nodes_perm")
        perm = nodes_perm.to(g.indptr.device, torch.int64).contiguous()
    elif algo == "rcmk":
        perm = rcmk_permutation(g, backend)
    elif algo == "degree":
        perm = degree_permutation(g)
    elif algo == "grow":
        perm = partition_permutation(grow_partition(g, k, seed=seed))
    elif algo == "metis":
        perm = partition_permutation(kway_partition(g, k, seed=seed))
    elif algo == "kway":
        perm = partition_permutation(kway_partition_device(g, k, seed=seed))
    else:
        raise RuntimeError("reorder_graph: unknown algorithm %r" % algo)
    return permute_graph(g, perm), perm


def recursive_metis_reorder(g: CSRGraph, partition_list, seed: int = 0, algo: str = "metis"
                            ) -> Tuple[CSRGraph, torch.Tensor]:
    """graphloader.py:358-372: one 'metis' reorder per entry of partition_list ([50, 60, 60] at
    :432), each applied to the graph the previous one produced.  algo="kway" partitions on the device
    instead.  Returns the final graph and the composed permutation (perm[i] = id in the ORIGINAL graph
    of final node i)."""
    if algo not in ("metis", "kway"):
        raise RuntimeError("recursive_metis_reorder: unknown algorithm %r (metis or kway)" % algo)
    perm = torch.arange(g.num_nodes, dtype=torch.int64, device=g.indptr.device)
    for level, k in enumerate(partition_list):
        g, p = reorder_graph(g, algo, k=int(k), seed=seed + level)
        perm = perm[p]
    return g, perm
