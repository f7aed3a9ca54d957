"""Worker of tests/test_gpu_sharded_inference.py (one process per GPU under torchrun): sage.ShardedInference
over real CUDA IPC mappings, against the single-GPU SAGE.inference / sage.evaluate that every rank also runs
on the whole graph."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "falcon-ttdforgnns_b200")]
import sage  # noqa: E402
from gnn_ops import aggregate_full  # noqa: E402

TOL = 1e-5
N = 20_000


def rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-300))


def model(dev, seed):
    torch.manual_seed(seed)
    m = sage.SAGE(N, 100, 128, 7, 3, 0.5, (16, 16), (28, 28, 28), (4, 5, 5), sparse=True,
                  learning_rate=0.05, embed_name="fbtt").to(dev)
    with torch.no_grad():
        for c in m.embed_layer.tt_cores:
            c.mul_(8.0)
    return m


def main():
    rank, world, local = (int(os.environ[k]) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    g = sage.synthetic_graph(N, 600_000, dev, seed=4)
    m = model(dev, 3)
    labels = torch.randint(0, 7, (N,), generator=torch.Generator().manual_seed(5)).to(dev)
    perm = torch.randperm(N, generator=torch.Generator().manual_seed(6)).to(dev)
    val_nid, test_nid = perm[:5000], perm[5000:9000]
    want = m.inference(g)
    val_ref, test_ref, _ = sage.evaluate(m, g, labels, val_nid, test_nid)
    uneven = [0, 0, N] if world == 2 else None          # rank 0 owns nothing
    for bounds in (None, uneven):
        inf = sage.ShardedInference(m, g, bounds=bounds)
        lo, hi = inf.lo, inf.hi
        got = inf.inference()
        assert got.shape == (hi - lo, 7)
        if hi > lo:
            assert rel(got, want[lo:hi]) < TOL, rel(got, want[lo:hi])
            assert torch.equal(got.argmax(1), want[lo:hi].argmax(1))
        # the layer-0 mean through the real mappings: every rank's rows written, then read across the node
        F = m.layers[0].in_feats
        inf._write(inf._IN)
        x = inf._own(inf._IN, F)
        full_x = m._all_rows(N)
        x.copy_(full_x[lo:hi])
        mean = inf._mean(inf._IN, F).clone()
        inf._barrier()
        assert torch.equal(mean, aggregate_full(g, full_x)[lo:hi])
        val, test = inf.evaluate(labels, val_nid, test_nid)
        assert (val, test) == (val_ref, test_ref), ((val, test), (val_ref, test_ref))
        both = [None] * world
        dist.all_gather_object(both, (val, test))
        assert all(b == both[0] for b in both)
        inf.close()
    # different parameters: every rank raises
    other = model(dev, 3 + rank)
    try:
        sage.ShardedInference(other, g)
        raise AssertionError("different parameters were accepted")
    except RuntimeError as e:
        assert "different parameters" in str(e)
    # close() followed by a new ShardedInference works
    inf = sage.ShardedInference(m, g)
    assert rel(inf.inference(), want[inf.lo:inf.hi]) < TOL
    inf.close()
    dist.barrier()
    if rank == 0:
        print("SHARDED_INFERENCE_OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
