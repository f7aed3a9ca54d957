"""Whole-graph mean aggregation (ttg_mean_agg_plan / ttg_mean_agg) without a GPU: the size queries and the
argument checks of the C ABI, all of which happen before any CUDA call."""
import ctypes

FAKE = ctypes.c_void_p(256)     # never dereferenced: every call below fails its checks first


def test_mean_agg_size_queries(ttg_lib):
    lib = ttg_lib
    for n, e in ((-1, 10), (1 << 31, 10), (10, -1), (10, (1 << 37) + 1)):
        assert lib.ttg_mean_agg_plan_bytes(n, e) == 0
        assert lib.ttg_mean_agg_workspace_bytes(n, e, 4) == 0
    for F in (0, -3):
        assert lib.ttg_mean_agg_workspace_bytes(100, 1000, F) == 0
    a = lib.ttg_mean_agg_plan_bytes(1000, 50000)
    assert a == lib.ttg_mean_agg_plan_bytes(1000, 50000)
    # N + E / 256 items of 16 bytes
    assert a >= 16 * (1000 + 50000 // 256)
    assert lib.ttg_mean_agg_plan_bytes(2000, 50000) > a
    assert lib.ttg_mean_agg_plan_bytes(1000, 500000) > a
    assert lib.ttg_mean_agg_plan_bytes(0, 0) > 0 and lib.ttg_mean_agg_plan_bytes(1, 0) > 0
    w = lib.ttg_mean_agg_workspace_bytes(1000, 500000, 47)
    assert w == lib.ttg_mean_agg_workspace_bytes(1000, 500000, 47)
    # partial rows of the nodes with more than 256 in-edges: fewer than 2 E / 256 of them
    assert w >= 4 * 47 * (500000 // 256 + 500000 // 257)
    assert lib.ttg_mean_agg_workspace_bytes(1000, 500000, 256) > w
    assert lib.ttg_mean_agg_workspace_bytes(1, 0, 1) > 0
    # papers100M shape is sized, not refused
    assert lib.ttg_mean_agg_plan_bytes(111_059_956, 1_615_685_872) > 16 * 111_059_956


def test_mean_agg_plan_refuses_bad_arguments(ttg_lib):
    lib = ttg_lib
    pb = lib.ttg_mean_agg_plan_bytes(100, 400)
    wb = lib.ttg_mean_agg_workspace_bytes(100, 400, 1)

    def call(n=100, e=400, indptr=FAKE, plan=FAKE, plan_bytes=pb, ws=FAKE, ws_bytes=wb):
        return lib.ttg_mean_agg_plan(n, e, indptr, plan, plan_bytes, ws, ws_bytes, None)

    for n in (-1, 1 << 31):
        assert call(n=n) == -1 and b"num_nodes" in lib.ttg_last_error()
    assert call(e=-1) == -1 and b"num_edges" in lib.ttg_last_error()
    assert call(indptr=None) == -1 and b"null pointer" in lib.ttg_last_error()
    assert call(plan=None) == -1 and b"null pointer" in lib.ttg_last_error()
    assert call(plan=ctypes.c_void_p(264)) == -1 and b"aligned" in lib.ttg_last_error()
    assert call(plan_bytes=pb - 1) == -3 and b"plan buffer" in lib.ttg_last_error()
    assert call(ws=None) == -3 and b"workspace" in lib.ttg_last_error()
    assert call(ws_bytes=wb - 1) == -3 and b"workspace" in lib.ttg_last_error()
    assert call(n=1000) == -3             # more nodes than the plan was sized for


def test_mean_agg_refuses_bad_arguments(ttg_lib):
    lib = ttg_lib
    pb = lib.ttg_mean_agg_plan_bytes(100, 40000)
    wb = lib.ttg_mean_agg_workspace_bytes(100, 40000, 47)

    def call(n=100, e=40000, F=47, indptr=FAKE, indices=FAKE, plan=FAKE, plan_bytes=pb, x=FAKE, out=FAKE, ws=FAKE,
             ws_bytes=wb):
        return lib.ttg_mean_agg(n, e, F, indptr, indices, plan, plan_bytes, x, out, ws, ws_bytes, None)

    for F in (0, -1):
        assert call(F=F) == -1 and b"F=" in lib.ttg_last_error()
    for n in (-1, 1 << 31):
        assert call(n=n) == -1 and b"num_nodes" in lib.ttg_last_error()
    assert call(e=-5) == -1 and b"num_edges" in lib.ttg_last_error()
    for name in ("indptr", "indices", "plan", "x", "out"):
        assert call(**{name: None}) == -1 and b"null pointer" in lib.ttg_last_error(), name
    assert call(plan=ctypes.c_void_p(260)) == -1 and b"aligned" in lib.ttg_last_error()
    assert call(plan_bytes=pb - 1) == -3 and b"plan buffer" in lib.ttg_last_error()
    assert call(ws=None) == -3 and b"workspace" in lib.ttg_last_error()
    assert call(ws_bytes=wb - 1) == -3 and b"workspace" in lib.ttg_last_error()
    assert call(F=256) == -3              # a workspace sized for 47 columns is short for 256
    assert call(e=400000) == -3           # more edges than the plan was sized for
