"""sage.ShardedInference against single-GPU SAGE.inference, one command per world size under torchrun:

    python -m torch.distributed.run --nproc-per-node W profiles/tools/sharded_inference_time.py [--reps 5]
        [--out profiles/r2i_sharded_inference.jsonl] [--papers]

Rank 0 appends JSON lines to --out, each naming the card and its power limit read in the same command:
  * products-shaped power-law graph (sage.synthetic_graph, 2.45 M nodes, 123.7 M edges), model 100 -> 256 -> 256
    -> 47 (fbtt, (125, 140, 140) x (4, 5, 5), rank 16): SAGE.inference on one GPU (rank 0, the whole graph) as the
    baseline, the sharded inference end to end (slowest rank, median of --reps), the per-layer barrier,
    aggregation and GEMM times from events, the logits' largest relative difference to the baseline, and the
    remote bytes the sharded means read (cross-shard edges x F x 4, counted from the graph) with the NVLink read
    rate they imply over the aggregation time;
  * 125-community graph (2.45 M nodes, 24 M edges): default bounds against the graph reordered by
    reorder_graph(g, "kway", W) with the part bounds (W > 1);
  * --papers, eight ranks only: 111,059,956 nodes, 1.6 B edges, (481, 481, 481) x (4, 4, 8) rank-32 table,
    128 -> 256 -> 256 -> 172: seconds per layer and peak device bytes per rank, the graph compared by checksum
    across ranks."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for _p in (ROOT, os.path.join(ROOT, "falcon-ttdforgnns_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name(0)
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0)


def cross_edges(g, bounds):
    """In-edges whose source lives in another shard than the destination."""
    owner = lambda ids: torch.bucketize(ids, torch.tensor(bounds[1:-1], device=ids.device), right=True)
    dst = torch.repeat_interleave(torch.arange(g.num_nodes, device=g.indptr.device), g.indptr[1:] - g.indptr[:-1])
    return int((owner(dst) != owner(g.indices.long())).sum())


def timed(fn, reps):
    """Median seconds of fn() over reps calls, each ended by a synchronise and, across ranks, by the slowest."""
    ts = []
    for _ in range(reps):
        dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        t = torch.tensor([a.elapsed_time(b) / 1e3], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ts.append(float(t))
    return statistics.median(ts), min(ts), max(ts)


def phases(inf, model):
    """Seconds per layer of barrier, aggregation and GEMM (fc_neigh before the mean counts as GEMM) on this rank."""
    inf.events = []
    inf.inference()
    torch.cuda.synchronize()
    ev, inf.events = inf.events, None
    out, layer, prev = [], None, ev[1][1]          # after "rows"
    for tag, e in ev[2:]:
        if layer is None:
            layer = {"barrier_s": 0.0, "aggregate_s": 0.0, "gemm_s": 0.0}
        layer[tag + "_s"] = layer[tag + "_s"] + prev.elapsed_time(e) / 1e3
        prev = e
        if tag == "gemm" and "agg_done" in layer:
            out.append({k: round(v, 6) for k, v in layer.items() if k != "agg_done"})
            layer = None
        elif tag == "aggregate":
            layer["agg_done"] = 1
    assert len(out) == len(model.layers)
    return out


def run(name, g, model, bounds_list, reps, out, base, info, world, rank):
    import sage
    for label, bounds in bounds_list:
        inf = sage.ShardedInference(model, g, bounds=bounds)
        inf.inference()
        t = timed(inf.inference, reps)
        got = inf.inference()
        lay = phases(inf, model)
        diff = None
        if base is not None:
            want = base[inf.lo:inf.hi]
            d = torch.tensor([float((got.double() - want.double()).abs().max()) if got.numel() else 0.0],
                             device="cuda")
            dist.all_reduce(d, op=dist.ReduceOp.MAX)
            diff = float(d) / float(base.abs().max())
        lays = [None] * world
        dist.all_gather_object(lays, lay)
        cross = cross_edges(g, inf.bounds)
        if rank == 0:
            agg = [max(l[i]["aggregate_s"] for l in lays) for i in range(len(model.layers))]
            widths = [min(c.in_feats, c.out_feats) for c in model.layers]
            rec = {"gpu": info, "world": world, "graph": name, "bounds": label, "shard_rows": [
                inf.bounds[r + 1] - inf.bounds[r] for r in range(world)], "sharded_median_s": round(t[0], 5),
                "sharded_min_s": round(t[1], 5), "sharded_max_s": round(t[2], 5), "reps": reps,
                "layers_rank0": lays[0], "aggregate_s_slowest_rank": [round(a, 6) for a in agg],
                "cross_shard_edges": cross, "edges": g.num_edges,
                "remote_bytes_per_layer": [cross * w * 4 for w in widths],
                "remote_GBps_per_layer": [round(cross * w * 4 / a / 1e9, 1) if cross and a > 0 else None
                                          for w, a in zip(widths, agg)],
                "max_rel_diff_to_single_gpu": diff,
                "peak_torch_bytes_rank0": torch.cuda.max_memory_allocated(), "peer_buffer_bytes": 3 * inf.region_bytes}
            with open(out, "a") as f:
                f.write(json.dumps(rec) + "\n")
            print(json.dumps(rec), flush=True)
        inf.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r2i_sharded_inference.jsonl"))
    ap.add_argument("--papers", action="store_true")
    args = ap.parse_args()
    rank, world, local = (int(os.environ[k]) for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    import reorder
    import sage
    info = gpu_info()
    n, e = 2_449_029, 123_718_280
    torch.manual_seed(0)
    model = sage.SAGE(n, 100, 256, 47, 3, 0.5, (16, 16), (125, 140, 140), (4, 5, 5), sparse=True,
                      learning_rate=0.01, embed_name="fbtt").to(dev)
    if not args.papers:
        g = sage.synthetic_graph(n, e, dev, seed=0)
        base = model.inference(g)
        t = timed(lambda: model.inference(g), args.reps)
        if rank == 0:
            rec = {"gpu": info, "world": world, "graph": "synthetic_graph(%d, %d, seed=0)" % (n, e),
                   "what": "SAGE.inference, one GPU, whole graph (baseline)", "median_s": round(t[0], 5),
                   "min_s": round(t[1], 5), "max_s": round(t[2], 5), "reps": args.reps}
            with open(args.out, "a") as f:
                f.write(json.dumps(rec) + "\n")
            print(json.dumps(rec), flush=True)
        run("powerlaw", g, model, [("default", None)], args.reps, args.out, base, info, world, rank)
        del g, base
        gc, _ = sage.synthetic_community_graph(n, 24_000_000, 125, 0.9, dev, seed=0)
        cases = [("default", None)]
        if world > 1:
            labels = reorder.kway_partition_device(gc, world)        # the partition reorder_graph lays out
            sizes = torch.bincount(labels.long(), minlength=world).cumsum(0).tolist()
            gk, _ = reorder.reorder_graph(gc, "kway", world)
            cases_k = [("kway parts", [0] + sizes)]
        run("community125", gc, model, cases, args.reps, args.out, None, info, world, rank)
        if world > 1:
            run("community125 kway-reordered", gk, model, cases_k, args.reps, args.out, None, info, world, rank)
    else:
        if world != 8:
            raise SystemExit("--papers runs on eight ranks")
        N, E = 111_059_956, 1_615_685_872
        g = sage.synthetic_graph(N, E, dev, seed=0)
        s = torch.tensor([int(g.indptr[::4096].sum()), int(g.indices[::4096].long().sum())], device=dev)
        ss = [torch.empty_like(s) for _ in range(world)]
        dist.all_gather(ss, s)
        assert all(torch.equal(x, s) for x in ss), "ranks generated different graphs"
        torch.manual_seed(0)
        model = sage.SAGE(N, 128, 256, 172, 3, 0.5, (32, 32), (481, 481, 481), (4, 4, 8), sparse=True,
                          learning_rate=0.01, embed_name="fbtt").to(dev)
        torch.cuda.reset_peak_memory_stats()
        run("papers", g, model, [("default", None)], 1, args.out, None, info, world, rank)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
