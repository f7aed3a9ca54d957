"""Sharded full-neighbour inference without a device: the shard bounds of sage.ShardedInference (balanced
contiguous ranges, checked caller bounds) and the argument checks ttg_mean_agg_sharded makes before any CUDA
call."""
import ctypes as C

import pytest
import torch


def _indptr(deg):
    indptr = torch.zeros(len(deg) + 1, dtype=torch.int64)
    indptr[1:] = torch.cumsum(torch.as_tensor(deg, dtype=torch.int64), 0)
    return indptr


def _power_law_indptr(n, seed):
    gen = torch.Generator().manual_seed(seed)
    u = torch.rand(n, generator=gen, dtype=torch.float64)
    deg = ((1.0 - u).clamp_min(1e-9).pow(-1.0 / 1.5)).floor().to(torch.int64).clamp_max(5000)
    return _indptr(deg)


@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("seed", [0, 1])
def test_default_bounds_cover_all_nodes_and_balance_the_weight(world, seed):
    import sage
    indptr = _power_law_indptr(20_000, seed)
    n, e = indptr.numel() - 1, int(indptr[-1])
    b = sage.shard_bounds(indptr, world)
    assert len(b) == world + 1 and b[0] == 0 and b[-1] == n
    assert all(b[r] <= b[r + 1] for r in range(world))
    c = -(-e // n)
    weight = (indptr[1:] - indptr[:-1]) + c
    ideal = float(weight.sum()) / world
    heaviest = int(weight.max())
    for r in range(world):
        w = int(weight[b[r]:b[r + 1]].sum())
        assert abs(w - ideal) <= heaviest + 1, (r, w, ideal, heaviest)
    assert sage.shard_bounds(indptr, world) == b               # a function of indptr alone


def test_more_ranks_than_nodes_gives_empty_shards():
    import sage
    indptr = _indptr([3, 0, 5])
    b = sage.shard_bounds(indptr, 8)
    assert len(b) == 9 and b[0] == 0 and b[-1] == 3
    assert all(b[r] <= b[r + 1] for r in range(8))
    sizes = [b[r + 1] - b[r] for r in range(8)]
    assert sum(sizes) == 3 and sizes.count(0) >= 5 and max(sizes) == 1
    assert sage.shard_bounds(_indptr([]), 4) == [0, 0, 0, 0, 0]


def test_caller_bounds_are_checked():
    import sage
    assert sage.check_bounds([0, 4, 4, 10], 10, 3) == [0, 4, 4, 10]      # an empty shard is fine
    for bad in ([1, 4, 4, 10], [0, 4, 4, 9], [0, 6, 4, 10], [0, 10]):     # start, end, decrease, count
        with pytest.raises(ValueError):
            sage.check_bounds(bad, 10, 3)


# ---- ttg_mean_agg_sharded refuses bad arguments before any CUDA call -----------------------------------------
FAKE = 1 << 20            # 16-byte aligned addresses that are never dereferenced


def _call(lib, world=2, bounds=(0, 5, 10), blocks=(FAKE, FAKE + 4096), ws_bytes=None, num_dst=5, num_edges=20, F=8):
    nb = max(len(bounds), 1)
    b = (C.c_int64 * nb)(*bounds)
    x = (C.c_void_p * max(len(blocks), 1))(*blocks)
    plan_bytes = lib.ttg_mean_agg_plan_bytes(num_dst, num_edges)
    need = lib.ttg_mean_agg_workspace_bytes(num_dst, num_edges, F)
    return lib.ttg_mean_agg_sharded(num_dst, num_edges, F, C.c_void_p(FAKE), C.c_void_p(FAKE), C.c_void_p(FAKE),
                                    plan_bytes, world, b, x, C.c_void_p(FAKE), C.c_void_p(FAKE),
                                    need if ws_bytes is None else ws_bytes, None)


def test_sharded_mean_refuses_bad_arguments(ttg_lib):
    lib = ttg_lib
    for world in (0, 9):
        assert _call(lib, world=world, bounds=[0] * 10, blocks=[FAKE] * 9) == -1
        assert b"world" in lib.ttg_last_error()
    assert _call(lib, bounds=(0, 7, 5)) == -1 and b"decrease" in lib.ttg_last_error()
    assert _call(lib, bounds=(1, 5, 10)) == -1 and b"bounds[0]" in lib.ttg_last_error()
    assert _call(lib, blocks=(FAKE, 0)) == -1 and b"null block 1" in lib.ttg_last_error()
    assert _call(lib, blocks=(FAKE, FAKE + 4)) == -1 and b"aligned" in lib.ttg_last_error()
    assert _call(lib, ws_bytes=16) != 0 and b"workspace" in lib.ttg_last_error()
    assert _call(lib, F=0) == -1
    # an empty block may be null; with nothing else wrong and no destination the call launches nothing
    assert _call(lib, bounds=(0, 0, 10), blocks=(0, FAKE), num_dst=0, num_edges=0) == 0
