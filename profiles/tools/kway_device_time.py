"""Multilevel k-way partition: the host partitioner (reorder.kway_partition, csrc/kway_host.cu) against the device
partitioner (reorder.kway_partition_device, csrc/kway.cu) on the same products-shaped graphs, partitioner seeds
0..2.  Prints one JSON line per (graph, seed): device seconds per phase (symmetrise, coarsening, host step,
refinement), levels and the coarsest graph, cut / planted cut (community graphs), cut / host cut, the largest
and smallest part against the bounds, peak device bytes, and the host seconds with the host / device ratio.
The first line names the card and its power limit.

    python profiles/tools/kway_device_time.py [--graphs community24m,community,powerlaw] [--seeds 3] [--first-seed 0] [--papers]

--papers adds the papers100M shape (111 M nodes, 1.6 B edges) on the device path alone."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

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


def cut_of(g, labels):
    dst = torch.repeat_interleave(torch.arange(g.num_nodes, device=labels.device), g.indptr[1:] - g.indptr[:-1])
    return int((labels[dst] != labels[g.indices.long()]).sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graphs", default="community24m,community,powerlaw")
    ap.add_argument("--seeds", type=int, default=3)
    ap.add_argument("--first-seed", type=int, default=0)
    ap.add_argument("--papers", action="store_true")
    ap.add_argument("--no-host", action="store_true")
    args = ap.parse_args()
    import reorder
    import sage
    dev = torch.device("cuda", 0)
    k, ub = 125, 1.03
    shapes = {
        "community24m": lambda: sage.synthetic_community_graph(2_449_029, 24_000_000, k, 0.9, dev, seed=0),
        "community": lambda: sage.synthetic_community_graph(2_449_029, 123_718_280, k, 0.9, dev, seed=0),
        "powerlaw": lambda: (sage.synthetic_graph(2_449_029, 123_718_280, dev, seed=0), None),
        "papers": lambda: (sage.synthetic_graph(111_059_956, 1_615_685_872, dev, seed=0), None),
    }
    names = [s for s in args.graphs.split(",") if s] + (["papers"] if args.papers else [])
    print(json.dumps({"gpu": gpu_info(), "k": k, "ubfactor": ub}), flush=True)
    for name in names:
        g, comm = shapes[name]()
        n, nnz = g.num_nodes, g.num_edges
        ideal = -(-n // k)
        maxpw, minpw = max(ideal, int(ub * ideal)), int((n // k) / ub)
        planted = cut_of(g, comm) if comm is not None else None
        reorder.kway_partition_device(g, k, seed=0)        # first call: module load, allocator warm-up
        for seed in range(args.first_seed, args.first_seed + args.seeds):
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats(dev)
            base = torch.cuda.memory_allocated(dev)
            st = {}
            t0 = time.perf_counter()
            part = reorder.kway_partition_device(g, k, seed=seed, stats=st)
            torch.cuda.synchronize()
            dev_s = time.perf_counter() - t0
            sizes = torch.bincount(part.long(), minlength=k)
            rec = {"graph": name, "nodes": n, "directed_edges": nnz, "seed": seed,
                   "device_s": round(dev_s, 3),
                   "device_phases_s": {p: round(st[p + "_s"], 3)
                                       for p in ("symmetrise", "coarsen", "host_initial", "refine")},
                   "levels": st["levels"], "coarsest_nodes": st["coarsest_nodes"],
                   "coarsest_edges": st["coarsest_edges"], "refine_iterations": st["refine_iterations"],
                   "exact_fills": st["exact_fills"], "cut": st["cut"],
                   "largest_part": int(sizes.max()), "bound_max": maxpw,
                   "smallest_part": int(sizes.min()), "bound_min": minpw,
                   "bound_held": bool(sizes.max() <= maxpw and sizes.min() >= minpw),
                   "peak_device_bytes": torch.cuda.max_memory_allocated(dev) - base}
            if planted is not None:
                rec["planted_cut"] = planted
                rec["cut_over_planted"] = round(st["cut"] / planted, 4)
            if name != "papers" and not args.no_host:
                t0 = time.perf_counter()
                hpart, hcut = reorder.kway_partition(g, k, seed=seed, return_cut=True)
                rec["host_s"] = round(time.perf_counter() - t0, 2)
                rec["host_cut"] = hcut
                rec["cut_over_host_cut"] = round(st["cut"] / hcut, 4)
                rec["host_over_device_time"] = round(rec["host_s"] / dev_s, 1)
                if planted is not None:
                    rec["host_cut_over_planted"] = round(hcut / planted, 4)
            print(json.dumps(rec), flush=True)
            del part
        del g, comm
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
