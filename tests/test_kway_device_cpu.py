"""The device k-way partitioner's argument checks that need no device: "kway" without k and an unknown algorithm of
recursive_metis_reorder fail before the graph is touched (the graph here is None)."""
import pytest


def test_kway_needs_k():
    import reorder
    with pytest.raises(RuntimeError, match="needs k"):
        reorder.reorder_graph(None, "kway")


def test_kway_takes_no_backend():
    import reorder
    with pytest.raises(RuntimeError, match="applies to 'rcmk' only"):
        reorder.reorder_graph(None, "kway", k=4, backend="device")


def test_recursive_reorder_refuses_unknown_algorithm():
    import reorder
    with pytest.raises(RuntimeError, match="unknown algorithm"):
        reorder.recursive_metis_reorder(None, [4, 6], algo="grow")
