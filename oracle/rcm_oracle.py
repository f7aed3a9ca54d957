"""Reverse Cuthill-McKee order restated level by level, in numpy: the contract of csrc/rcm.cu.

    perm = rcm_order(indptr, indices)      # == scipy.sparse.csgraph.reverse_cuthill_mckee(adj, False)

adj is the CSR of the graph's in-neighbour lists (row v = in-list of v), as reorder.rcmk_permutation
builds it.  scipy runs a BFS with an insertion sort per parent; the same order, stated so that every
level can be computed at once:

1. sym_lists: scipy's adj + adj^T.  Canonical input (every in-list strictly increasing): row i holds
   the distinct neighbours of i ascending.  Any other input (sparsetools' general path): row i = the
   in-list of i as stored followed by every v with i in in-list(v) in increasing v (once per
   occurrence); the distinct entries in REVERSE order of first appearance.
2. degree: row length, + 1 if the row holds its own node (self loop); int32.
3. seed ranks: numpy.argsort of the degrees (scipy's own call; its tie order is numpy's).
4. components in increasing rank of their seed, the node of smallest rank.
5. level L + 1 of a component: every unvisited neighbour j of level f[0..m) is owned by the smallest
   (p, k), p the parent's position in f, k the position of j in the parent's row; the owned nodes
   sorted by (p, degree(j), k).
6. the levels of the components concatenated, reversed.

Out of contract: 128 or more parallel edges between one pair of nodes (scipy's int8 sum can wrap to 0
and drop the entry).  Test infrastructure only; the package never imports it.
"""
import numpy as np


def sym_lists(indptr, indices):
    """(sym_indptr int64, sym_indices int64) of scipy's adj + adj^T, rows ordered as scipy orders them."""
    n = indptr.shape[0] - 1
    rows = [indices[indptr[i]:indptr[i + 1]].tolist() for i in range(n)]
    canonical = all(all(r[k] < r[k + 1] for k in range(len(r) - 1)) for r in rows)
    tr = [[] for _ in range(n)]
    for v in range(n):
        for u in rows[v]:
            tr[u].append(v)
    out = []
    for i in range(n):
        first = dict.fromkeys(rows[i] + tr[i])          # distinct, in order of first appearance
        out.append(sorted(first) if canonical else list(first)[::-1])
    ptr = np.zeros(n + 1, np.int64)
    ptr[1:] = np.cumsum([len(r) for r in out])
    ind = np.array([j for r in out for j in r], np.int64)
    return ptr, ind


def degrees(ptr, ind):
    n = ptr.shape[0] - 1
    deg = np.diff(ptr).astype(np.int32)
    for i in range(n):
        if np.any(ind[ptr[i]:ptr[i + 1]] == i):
            deg[i] += 1
    return deg


def rcm_order(indptr, indices, return_stats=False):
    """perm (int64): new node i = old node perm[i].  return_stats: also (levels, components), levels
    counted as the most any component has."""
    indptr = np.asarray(indptr, np.int64)
    indices = np.asarray(indices)
    n = indptr.shape[0] - 1
    ptr, ind = sym_lists(indptr, indices)
    deg = degrees(ptr, ind)
    visited = np.zeros(n, bool)
    order, levels, components = [], 0, 0
    for seed in np.argsort(deg):                          # components in increasing seed rank
        if visited[seed]:
            continue
        components += 1
        visited[seed] = True
        front, depth = [int(seed)], 1
        order.append(int(seed))
        while front:
            owner = {}
            for p, u in enumerate(front):
                for k in range(ptr[u + 1] - ptr[u]):
                    j = int(ind[ptr[u] + k])
                    if not visited[j] and j not in owner:  # (p, k) increase along this walk: first = smallest
                        owner[j] = (p, k)
            front = sorted(owner, key=lambda j: (owner[j][0], deg[j], owner[j][1]))
            visited[front] = True
            order.extend(front)
            depth += bool(front)
        levels = max(levels, depth)
    perm = np.array(order[::-1], np.int64)
    return (perm, (levels, components)) if return_stats else perm


# ---- the graph families the contract is checked on ------------------------------------------------------
FAMILIES = ("canonical", "general", "parallel", "self_loops", "isolated", "tiny", "components", "ties")


def csr_from_edges(n, src, dst, canonical):
    """In-neighbour CSR of the edges src -> dst: sorted distinct in-lists (canonical) or the given order."""
    src, dst = np.asarray(src, np.int64), np.asarray(dst, np.int64)
    if canonical:
        pairs = np.unique(dst * n + src)
        dst, src = pairs // n, pairs % n
    else:
        o = np.argsort(dst, kind="stable")
        src, dst = src[o], dst[o]
    indptr = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(dst, minlength=n), out=indptr[1:])
    return indptr, src.astype(np.int32)


def random_case(rng, t):
    """Graph number t of a seeded sequence cycling through FAMILIES: (family, indptr, indices)."""
    kind = FAMILIES[t % len(FAMILIES)]
    n = int(rng.integers(2, 150))
    canonical = bool(rng.integers(0, 2))
    if kind == "canonical" or kind == "general":
        m = int(rng.integers(0, 3 * n))
        src, dst = rng.integers(0, n, m), rng.integers(0, n, m)
        canonical = kind == "canonical"
    elif kind == "parallel":                      # every edge 1..6 times, lists shuffled
        m = int(rng.integers(1, 2 * n))
        rep = rng.integers(1, 7, m)
        src, dst = np.repeat(rng.integers(0, n, m), rep), np.repeat(rng.integers(0, n, m), rep)
        o = rng.permutation(src.shape[0])
        src, dst, canonical = src[o], dst[o], False
    elif kind == "self_loops":
        m = int(rng.integers(0, 2 * n))
        loops = rng.choice(n, int(rng.integers(1, n + 1)), replace=False)
        src = np.concatenate([rng.integers(0, n, m), loops])
        dst = np.concatenate([rng.integers(0, n, m), loops])
    elif kind == "isolated":                      # most nodes without any edge
        n = int(rng.integers(20, 300))
        m = int(rng.integers(0, n // 4 + 1))
        src, dst = rng.integers(0, n, m), rng.integers(0, n, m)
    elif kind == "tiny":                          # 1-node graphs (with or without a self loop), 0-edge graphs
        n = int(rng.integers(1, 4)) if t % 16 < 8 else n
        m = int(rng.integers(0, 2)) if n == 1 else 0
        src, dst = np.zeros(m, np.int64), np.zeros(m, np.int64)
    elif kind == "components":                    # many small pieces under scrambled ids
        sizes = rng.integers(1, 6, int(rng.integers(10, 60)))
        n = int(sizes.sum())
        base = np.concatenate([[0], np.cumsum(sizes)[:-1]])
        src, dst = [], []
        for b, s in zip(base, sizes):
            k = int(rng.integers(0, 2 * s))
            src.append(b + rng.integers(0, s, k))
            dst.append(b + rng.integers(0, s, k))
        scr = rng.permutation(n)
        src, dst = scr[np.concatenate(src)], scr[np.concatenate(dst)]
    else:                                         # "ties": unions of cycles, every degree equal
        scr = rng.permutation(n)
        a = np.arange(n)
        nxt = np.where(a % 10 == 9, a - 9, a + 1)
        nxt = np.where(nxt >= n, a - a % 10, nxt)
        src, dst = scr[a], scr[nxt]
        if not canonical:
            src, dst = np.concatenate([src, dst]), np.concatenate([dst, src])
            o = rng.permutation(src.shape[0])
            src, dst = src[o], dst[o]
    indptr, indices = csr_from_edges(n, src, dst, canonical)
    return kind, indptr, indices
