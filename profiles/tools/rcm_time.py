"""Reverse Cuthill-McKee: scipy (reorder_graph(g, "rcmk"), DGL's 'rcmk') against the device path
(backend="device", csrc/rcm.cu) on products-shaped graphs.  Asserts that the two permutations are
identical and prints one JSON line per graph: the seconds of each device phase (symmetrise, host
argsort, components, BFS, final order, relabelling), the scipy seconds, BFS levels and components.

    python profiles/tools/rcm_time.py [--graphs powerlaw,community] [--papers]

--papers adds the papers100M shape (111 M nodes, 1.6 B edges) on the device path alone (scipy would
have to build a 3.2 B-entry symmetric CSR in host memory); it states the device bytes it needs first."""
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


def timed_device(g, reorder):
    torch.cuda.synchronize()
    st = {}
    t0 = time.perf_counter()
    perm = reorder.rcmk_permutation(g, backend="device", stats=st)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    g2 = reorder.permute_graph(g, perm)
    torch.cuda.synchronize()
    st["permute_s"] = time.perf_counter() - t1
    st["rcm_total_s"] = t1 - t0
    return perm, g2, st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--graphs", default="powerlaw,community")
    ap.add_argument("--papers", action="store_true")
    args = ap.parse_args()
    import _ttg
    import reorder
    import sage
    dev = torch.device("cuda", 0)
    lib = _ttg.lib()
    shapes = {"powerlaw": lambda: sage.synthetic_graph(2_449_029, 123_718_280, dev, seed=0),
              "community": lambda: sage.synthetic_community_graph(2_449_029, 24_000_000, 125, 0.9, dev, seed=0)[0]}
    names = [s for s in args.graphs.split(",") if s]
    if args.papers:
        names.append("papers")
        shapes["papers"] = lambda: sage.synthetic_graph(111_059_956, 1_615_685_872, dev, seed=0)
    gpu = gpu_info()
    for name in names:
        g = shapes[name]()
        n, nnz = g.num_nodes, g.num_edges
        ws = lib.ttg_rcm_symmetrise_workspace_bytes(n, nnz)
        need = {"symmetrise_workspace": ws, "sym_indices": 8 * nnz, "sym_indptr": 8 * (n + 1),
                "order_workspace": lib.ttg_rcm_order_workspace_bytes(n)}
        # stated before the run, so that a run that does not fit still leaves the number behind
        print(json.dumps({"graph": name, "nodes": n, "directed_edges": nnz, "device_bytes_needed": need,
                          "graph_bytes": 8 * (n + 1) + 4 * nnz,
                          "device_free_bytes": torch.cuda.mem_get_info(dev)[0]}), flush=True)
        rec = {"graph": name, "nodes": n, "directed_edges": nnz, "gpu": gpu, "device_bytes": need}
        timed_device(g, reorder)                         # first call: module load, allocations
        perm, g2, st = timed_device(g, reorder)
        rec["device"] = {k: (round(v, 4) if isinstance(v, float) else v) for k, v in st.items()}
        if name != "papers":
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            want = reorder.rcmk_permutation(g)
            torch.cuda.synchronize()
            rec["scipy_s"] = round(time.perf_counter() - t0, 3)
            assert torch.equal(perm, want), "device and scipy permutations differ"
            rec["identical_permutation"] = True
            rec["speedup_vs_scipy"] = round(rec["scipy_s"] / (st["rcm_total_s"]), 1)
        else:
            rec["identical_permutation"] = None      # scipy not run at this size
            assert torch.equal(torch.sort(perm).values, torch.arange(n, device=dev))
        print(json.dumps(rec), flush=True)
        del g, g2, perm
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
