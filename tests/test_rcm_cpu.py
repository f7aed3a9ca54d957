"""Reverse Cuthill-McKee without a GPU: the level-synchronous restatement (oracle/rcm_oracle.py, the
contract of csrc/rcm.cu) against scipy, and the argument checks of the C ABI."""
import ctypes

import numpy as np
import pytest
from scipy import sparse
from scipy.sparse.csgraph import reverse_cuthill_mckee

from oracle import rcm_oracle as ro


def _scipy_rcm(indptr, indices):
    n = indptr.shape[0] - 1
    adj = sparse.csr_matrix((np.ones(indices.shape[0], np.int8), indices, indptr), shape=(n, n))
    return reverse_cuthill_mckee(adj, symmetric_mode=False)


def test_oracle_is_scipys_order_on_every_family():
    rng = np.random.default_rng(2024)
    seen = {k: 0 for k in ro.FAMILIES}
    canonical = general = 0
    for t in range(480):
        kind, indptr, indices = ro.random_case(rng, t)
        want = _scipy_rcm(indptr, indices)
        got = ro.rcm_order(indptr, indices)
        assert np.array_equal(got, want), (t, kind)
        seen[kind] += 1
        lists = [indices[indptr[i]:indptr[i + 1]] for i in range(indptr.shape[0] - 1)]
        if all(np.all(np.diff(r) > 0) for r in lists):
            canonical += 1
        else:
            general += 1
    assert min(seen.values()) == 60 and canonical > 100 and general > 100


def test_oracle_edge_cases():
    one = np.array([0, 0], np.int64), np.zeros(0, np.int32)
    assert ro.rcm_order(*one).tolist() == [0]
    loop = np.array([0, 1], np.int64), np.zeros(1, np.int32)
    assert ro.rcm_order(*loop).tolist() == [0]
    empty = np.zeros(6, np.int64), np.zeros(0, np.int32)
    assert np.array_equal(ro.rcm_order(*empty), _scipy_rcm(*empty))
    # a path 0 - 1 - 2 - 3: one component, four levels
    ip, ix = ro.csr_from_edges(4, [0, 1, 1, 2, 2, 3], [1, 0, 2, 1, 3, 2], True)
    perm, (levels, comps) = ro.rcm_order(ip, ix, return_stats=True)
    assert np.array_equal(perm, _scipy_rcm(ip, ix)) and (levels, comps) == (4, 1)


def test_non_canonical_rows_are_in_reverse_order_of_first_appearance():
    # in-list of 0 = [2, 1] (unsorted) and 1 -> 2: row 0 = [2, 1] ++ [] reversed -> [1, 2]
    ip, ix = np.array([0, 2, 2, 3], np.int64), np.array([2, 1, 1], np.int32)
    ptr, ind = ro.sym_lists(ip, ix)
    assert ind[ptr[0]:ptr[1]].tolist() == [1, 2]
    assert ind[ptr[2]:ptr[3]].tolist() == [0, 1]      # [1] ++ [0] reversed
    assert ind[ptr[1]:ptr[2]].tolist() == [2, 0]      # [] ++ [0, 2] reversed


# ---- C ABI ----------------------------------------------------------------------------------------------
FAKE = ctypes.c_void_p(256)     # never dereferenced: every call below fails its checks first


def test_rcm_workspace_queries(ttg_lib):
    lib = ttg_lib
    assert lib.ttg_rcm_symmetrise_workspace_bytes(0, 0) == 0
    assert lib.ttg_rcm_symmetrise_workspace_bytes(1 << 31, 0) == 0
    assert lib.ttg_rcm_symmetrise_workspace_bytes(10, -1) == 0
    assert lib.ttg_rcm_order_workspace_bytes(0) == 0
    assert lib.ttg_rcm_order_workspace_bytes(1 << 31) == 0
    a = lib.ttg_rcm_symmetrise_workspace_bytes(1000, 5000)
    assert a == lib.ttg_rcm_symmetrise_workspace_bytes(1000, 5000)
    assert lib.ttg_rcm_symmetrise_workspace_bytes(1000, 10000) > a > 2 * 5000 * 24
    assert lib.ttg_rcm_symmetrise_workspace_bytes(1, 0) > 0
    assert lib.ttg_rcm_order_workspace_bytes(2000) > lib.ttg_rcm_order_workspace_bytes(1000) > 0
    # 64-bit entry counts: more than 2^31 symmetrised entries are sized, not refused
    assert lib.ttg_rcm_symmetrise_workspace_bytes(1 << 30, 3 << 30) > 6 * (1 << 30) * 24


def test_rcm_symmetrise_refuses_bad_arguments(ttg_lib):
    lib = ttg_lib
    out = ctypes.c_int64(-1)
    ws = lib.ttg_rcm_symmetrise_workspace_bytes(100, 400)

    def call(n, nnz, ptrs=(FAKE,) * 5, ws_ptr=FAKE, ws_bytes=ws, sym=ctypes.byref(out)):
        return lib.ttg_rcm_symmetrise(n, nnz, *ptrs, sym, ws_ptr, ws_bytes, None)

    for n in (0, -5, 1 << 31):
        assert call(n, 10) == -1 and b"num_nodes" in lib.ttg_last_error()
    assert call(100, -1) == -1
    for i in range(5):
        ptrs = [FAKE] * 5
        ptrs[i] = None
        assert call(100, 400, tuple(ptrs)) == -1 and b"null pointer" in lib.ttg_last_error()
    assert call(100, 400, sym=None) == -1
    assert call(100, 400, ws_ptr=None) == -3
    assert call(100, 400, ws_bytes=ws - 1) == -3 and b"workspace" in lib.ttg_last_error()
    assert lib.ttg_rcm_symmetrise_workspace_bytes(100, 4000) > ws
    assert call(100, 4000) == -3         # more entries than the workspace was sized for
    assert out.value == -1


def test_rcm_order_refuses_bad_arguments(ttg_lib):
    lib = ttg_lib
    ws = lib.ttg_rcm_order_workspace_bytes(100)

    def call(n, ptrs=(FAKE,) * 5, ws_ptr=FAKE, ws_bytes=ws, sym_edges=10):
        return lib.ttg_rcm_order(n, sym_edges, *ptrs, None, None, ws_ptr, ws_bytes, None)

    for n in (0, -1, 1 << 31):
        assert call(n) == -1 and b"num_nodes" in lib.ttg_last_error()
    assert call(100, sym_edges=-1) == -1
    for i in range(5):
        ptrs = [FAKE] * 5
        ptrs[i] = None
        assert call(100, tuple(ptrs)) == -1 and b"null pointer" in lib.ttg_last_error()
    assert call(100, ws_ptr=None) == -3
    assert call(100, ws_bytes=ws - 1) == -3 and b"workspace" in lib.ttg_last_error()
    assert lib.ttg_rcm_order_workspace_bytes(1000) > ws
    assert call(1000) == -3              # more nodes than the workspace was sized for


def test_backend_is_checked_before_the_graph_is_touched():
    import reorder
    with pytest.raises(RuntimeError, match="backend"):
        reorder.reorder_graph(None, "metis", k=4, backend="device")
    with pytest.raises(RuntimeError, match="backend"):
        reorder.reorder_graph(None, "degree", backend="device")
    with pytest.raises(RuntimeError, match="backend"):
        reorder.reorder_graph(None, "rcmk", backend="gpu")
    with pytest.raises(RuntimeError, match="backend"):
        reorder.rcmk_permutation(None, backend="cuda")
