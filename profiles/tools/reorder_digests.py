"""SHA-256 digests of what the device reordering code computes on seeded graphs, and the workspace sizes its
C ABI reports at the node and edge limits.  A change to csrc/rcm.cu, csrc/kway.cu, csrc/reorder.cu or reorder.py
that is meant to keep the outputs must keep every line this prints; tests/test_gpu_reorder_digests.py holds the
values and recomputes them.

Per graph: the input CSR, the device RCM permutation, ttg_kway_symmetrise's weighted CSR (xadj, adj, adjw, vw),
the device k-way labels for seeds 0-2 and k = 2, 7, 125 (where k <= N) with the stats that depend on the graph
and the seed alone, and permute_graph's relabelled CSR under the RCM permutation and under a seeded random one.

    python profiles/tools/reorder_digests.py [--out FILE]
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for _p in (ROOT, os.path.join(ROOT, "falcon-ttdforgnns_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

DEV = "cuda:0"
KWAY_K = (2, 7, 125)
KWAY_SEEDS = (0, 1, 2)
KWAY_STATS = ("levels", "coarsest_nodes", "coarsest_edges", "sym_edges", "refine_iterations", "exact_fills", "cut")


def _csr(n, src, dst):
    """in-neighbour lists: row dst holds src, in the given order"""
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
    lab = rng.permutation(n) % k
    src, dst = [], []
    for p in range(k):
        m = np.nonzero(lab == p)[0]
        src.append(rng.choice(m, size=m.shape[0] * deg_in // 2))
        dst.append(rng.choice(m, size=m.shape[0] * deg_in // 2))
    src.append(rng.integers(0, n, size=n * deg_out // 2))
    dst.append(rng.integers(0, n, size=n * deg_out // 2))
    s, d = np.concatenate(src), np.concatenate(dst)
    return _csr(n, np.concatenate([s, d]), np.concatenate([d, s]))


def _cliques():
    """two directed 4-cliques joined by one edge, a self loop, a duplicate edge and an isolated node"""
    edges = [(a, b) for a in range(4) for b in range(4) if a < b] + \
            [(a, b) for a in range(4, 8) for b in range(4, 8) if a < b] + [(3, 4), (2, 2), (0, 1)]
    return _csr(9, np.array([e[0] for e in edges]), np.array([e[1] for e in edges]))


def _hub(rng, n):
    """30 % isolated nodes and one node with a 100k-entry in-list and out-list"""
    live = rng.permutation(n)[: int(0.7 * n)]
    src, dst = rng.choice(live, size=600000), rng.choice(live, size=600000)
    hub = int(live[0])
    leaves = rng.choice(live, size=100000, replace=False)
    return _csr(n, np.concatenate([src, leaves, np.full(100000, hub)]),
                np.concatenate([dst, np.full(100000, hub), leaves]))


def _unsorted(rng, n, m):
    """in-lists in random order with duplicates and self loops"""
    src, dst = rng.integers(0, n, m), rng.integers(0, n, m)
    src = np.concatenate([src, src[: m // 10], np.arange(0, n, 7)])
    dst = np.concatenate([dst, dst[: m // 10], np.arange(0, n, 7)])
    o = rng.permutation(src.shape[0])
    return _csr(n, src[o], dst[o])


def graphs():
    """(name, CSRGraph on DEV) in a fixed order; every graph is generated from a seed"""
    import sage
    from oracle import rcm_oracle as ro
    from sampler import CSRGraph

    def dev(indptr, indices):
        return CSRGraph(torch.from_numpy(indptr).to(DEV), torch.from_numpy(indices).to(DEV))

    rng = np.random.default_rng(2026)
    for t in range(48):   # six of each family of the RCM oracle's cases (1-node and edgeless ones among them)
        kind, indptr, indices = ro.random_case(rng, t)
        yield "family%02d_%s" % (t, kind), dev(indptr, indices)
    yield "one_node", dev(np.zeros(2, np.int64), np.zeros(0, np.int32))
    yield "edgeless", dev(np.zeros(6, np.int64), np.zeros(0, np.int32))
    yield "cliques", dev(*_cliques())
    yield "grid64", dev(*_grid(64, 64))
    yield "unsorted", dev(*_unsorted(np.random.default_rng(11), 20000, 200000))
    yield "planted", dev(*_planted(np.random.default_rng(0), 20000, 50, 12, 2))
    yield "isolated_hub", dev(*_hub(np.random.default_rng(8), 300000))
    yield "community", sage.synthetic_community_graph(50000, 600000, 25, 0.9, torch.device(DEV), seed=1)[0]
    yield "powerlaw", sage.synthetic_graph(400000, 4_000_000, torch.device(DEV), seed=3)


class _Digest:
    def __init__(self):
        self.h = hashlib.sha256()

    def add(self, *items):
        for x in items:
            if isinstance(x, torch.Tensor):
                x = x.cpu().numpy()
            if isinstance(x, np.ndarray):
                x = np.ascontiguousarray(x)
                self.h.update(("%s%s" % (x.dtype.str, x.shape)).encode())
                self.h.update(x.tobytes())
            else:
                self.h.update(json.dumps(x, sort_keys=True).encode())
        return self

    def hex(self):
        return self.h.hexdigest()


def kway_symmetrise(g):
    import _ttg
    lib = _ttg.lib()
    n, nnz = g.num_nodes, int(g.indptr[-1])
    dev = g.indptr.device
    xadj = torch.empty(n + 1, dtype=torch.int64, device=dev)
    adj = torch.empty(max(2 * nnz, 1), dtype=torch.int32, device=dev)
    adjw = torch.empty(max(2 * nnz, 1), dtype=torch.int32, device=dev)
    vw = torch.empty(n, dtype=torch.int32, device=dev)
    m = C.c_int64(0)
    ws = torch.empty(lib.ttg_kway_symmetrise_workspace_bytes(n, nnz), dtype=torch.uint8, device=dev)
    _ttg.check(lib.ttg_kway_symmetrise(n, nnz, _ttg.ptr(g.indptr), _ttg.ptr(g.indices), _ttg.ptr(xadj),
                                       _ttg.ptr(adj), _ttg.ptr(adjw), _ttg.ptr(vw), C.byref(m), _ttg.ptr(ws),
                                       ws.numel(), _ttg.stream_of(dev)), "kway_symmetrise")
    return xadj, adj[:m.value], adjw[:m.value], vw


def graph_digests(name, g):
    """{"<name>/<what>": sha256} for one graph"""
    import reorder
    out = {name + "/input": _Digest().add(g.indptr, g.indices[:int(g.indptr[-1])]).hex()}
    perm = reorder.rcmk_permutation(g, backend="device")
    out[name + "/rcm"] = _Digest().add(perm).hex()
    out[name + "/kway_symmetrise"] = _Digest().add(*kway_symmetrise(g)).hex()
    d = _Digest()
    for k in KWAY_K:
        if k > g.num_nodes:
            continue
        for seed in KWAY_SEEDS:
            st = {}
            labels = reorder.kway_partition_device(g, k, seed=seed, stats=st)
            d.add(k, seed, labels, {s: st[s] for s in KWAY_STATS})
    out[name + "/kway"] = d.hex()
    rnd = torch.from_numpy(np.random.default_rng(g.num_nodes).permutation(g.num_nodes)).to(DEV)
    d = _Digest()
    for p in (perm, rnd):
        g2 = reorder.permute_graph(g, p)
        d.add(g2.indptr, g2.indices)
    out[name + "/permute"] = d.hex()
    return out


def family_digests(rows):
    """the 48 small family graphs fold into one digest per output, in graph order"""
    out, fold = {}, {}
    for key, value in rows.items():
        name, what = key.split("/")
        if name.startswith("family"):
            fold.setdefault("families/" + what, _Digest()).add(name, value)
        else:
            out[key] = value
    return dict({k: d.hex() for k, d in fold.items()}, **out)


def digests():
    torch.cuda.set_device(0)
    rows = {}
    for name, g in graphs():
        rows.update(graph_digests(name, g))
        del g
    return family_digests(rows)


# the node counts and edge counts on both sides of each limit of the C ABI
NODE_LIMITS = (2**31 - 2, 2**31 - 1, 2**31)
EDGE_LIMITS = (2**40, 2**40 + 1)


def workspace_sizes():
    """{"<query>(<args>)": bytes} at the limits; 0 means refused"""
    import _ttg
    lib = _ttg.lib()
    out = {}

    def q(fn, *args):
        out["%s(%s)" % (fn, ", ".join(str(a) for a in args))] = int(getattr(lib, fn)(*args))

    for n in NODE_LIMITS:
        q("ttg_rcm_symmetrise_workspace_bytes", n, 0)
        q("ttg_rcm_order_workspace_bytes", n)
        q("ttg_kway_symmetrise_workspace_bytes", n, 0)
        q("ttg_kway_coarsen_workspace_bytes", n, 0)
        q("ttg_kway_refine_workspace_bytes", n, 2)
        q("ttg_permute_csr_workspace_bytes", n)
    for e in EDGE_LIMITS:
        q("ttg_rcm_symmetrise_workspace_bytes", 1000, e)
        q("ttg_kway_symmetrise_workspace_bytes", 1000, e)
        q("ttg_kway_coarsen_workspace_bytes", 1000, e)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    t0 = time.perf_counter()
    rec = {"gpu": torch.cuda.get_device_name(0), "digests": digests(), "workspace_bytes": workspace_sizes(),
           "seconds": round(time.perf_counter() - t0, 1)}
    text = json.dumps(rec, indent=1, sort_keys=True)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
