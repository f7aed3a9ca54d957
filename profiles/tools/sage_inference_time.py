"""Full-neighbour GraphSAGE inference at products shape (2,449,029 nodes, 123.7 M edges, power-law in-degrees):
the whole-graph mean aggregation by the one-warp-per-destination kernel of sampled blocks (ttg_spmm_csr_fwd)
against the edge-balanced one (ttg_mean_agg) at F = 100, 256 and 47, the plan build, and SAGE.inference end to
end split per layer into rows, aggregation and dense layers.  One JSON line per measurement.

    python profiles/tools/sage_inference_time.py [--calls 30] [--warmup 3]

The two kernels are called alternately, each timed with CUDA events around one call; both read an [N, F]
input of 0.46 to 2.5 GB, far more than the 126 MB of L2.  The outputs must agree to 1e-5 relative to their
maximum.  The card's name and power limit are read with a read-only nvidia-smi query."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for _p in (ROOT, os.path.join(ROOT, "falcon-ttdforgnns_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name(0)
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0)


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def summary(ts):
    return {"median_ms": round(statistics.median(ts), 4), "min_ms": round(min(ts), 4),
            "max_ms": round(max(ts), 4), "calls": len(ts)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--widths", default="100,256,47")
    args = ap.parse_args()
    import _ttg
    import gnn_ops
    import sage
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _ttg.lib()
    gpu = gpu_info()
    g = sage.synthetic_graph(2_449_029, 123_718_280, dev, seed=0)
    n, e = g.num_nodes, g.num_edges
    deg = g.indptr[1:] - g.indptr[:-1]
    stream = _ttg.stream_of(dev)
    print(json.dumps({"gpu": gpu, "graph": "synthetic_graph(2449029, 123718280, seed=0)", "nodes": n, "edges": e,
                      "max_in_degree": int(deg.max()), "nodes_above_32": int((deg > 32).sum()),
                      "nodes_above_256": int((deg > 256).sum()), "nodes_above_1000": int((deg > 1000).sum()),
                      "edges_of_nodes_above_32": int(deg[deg > 32].sum())}), flush=True)

    # plan build (count, scan, scatter), on a graph object without a kept plan each time
    ts = []
    for i in range(args.warmup + 10):
        if hasattr(g, "_mean_agg_plan"):
            del g._mean_agg_plan
        t = event_ms(lambda: gnn_ops.mean_agg_plan(g))
        if i >= args.warmup:
            ts.append(t)
    plan = gnn_ops.mean_agg_plan(g)
    print(json.dumps({"gpu": gpu, "what": "plan_build", "plan_bytes": plan.numel(), **summary(ts)}), flush=True)

    for F in [int(f) for f in args.widths.split(",")]:
        x = torch.randn((n, F), device=dev, generator=torch.Generator(device=dev).manual_seed(F))
        old = torch.empty((n, F), device=dev)
        new = torch.empty((n, F), device=dev)
        ws_bytes = lib.ttg_mean_agg_workspace_bytes(n, e, F)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)

        def run_old():
            _ttg.check(lib.ttg_spmm_csr_fwd(n, F, _ttg.ptr(g.indptr), _ttg.ptr(g.indices), None, 1, _ttg.ptr(x),
                                            _ttg.ptr(old), stream), "spmm_csr_fwd")

        def run_new():
            _ttg.check(lib.ttg_mean_agg(n, e, F, _ttg.ptr(g.indptr), _ttg.ptr(g.indices), _ttg.ptr(plan),
                                        plan.numel(), _ttg.ptr(x), _ttg.ptr(new), _ttg.ptr(ws), ws_bytes, stream),
                       "mean_agg")

        for _ in range(args.warmup):
            run_old()
            run_new()
        t_old, t_new = [], []
        for _ in range(args.calls):
            t_old.append(event_ms(run_old))
            t_new.append(event_ms(run_new))
        err = float((new.double() - old.double()).abs().max() / old.double().abs().max())
        assert err < 1e-5, "outputs differ: %g" % err
        rerun = new.clone()
        run_new()
        torch.cuda.synchronize()
        # bytes the gather needs at least: every edge's source row and index, every output row, indptr
        need = e * (4 * F + 4) + n * (4 * F + 8)
        so, sn = summary(t_old), summary(t_new)
        print(json.dumps({"gpu": gpu, "what": "aggregation", "F": F, "spmm_csr_fwd": so, "mean_agg": sn,
                          "speedup_median": round(so["median_ms"] / sn["median_ms"], 2),
                          "mean_agg_GBps_of_needed_bytes": round(need / sn["median_ms"] / 1e6, 1),
                          "max_rel_diff": err, "mean_agg_repeat_bit_identical": bool(torch.equal(rerun, new)),
                          "workspace_bytes": ws_bytes}), flush=True)
        del x, old, new, ws, rerun
        torch.cuda.empty_cache()

    # SAGE.inference at bench_sage's model shape: 100 -> 256 -> 256 -> 47, TT table (125, 140, 140) x (4, 5, 5)
    torch.manual_seed(0)
    model = sage.SAGE(n, 100, 256, 47, 3, 0.5, (16, 16), (125, 140, 140), (4, 5, 5), sparse=True,
                      learning_rate=0.01, embed_name="fbtt").to(dev)
    model.eval()
    model.inference(g)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    ts = [event_ms(lambda: model.inference(g)) for _ in range(5)]
    peak = torch.cuda.max_memory_allocated(dev) - base
    # the same steps one by one (SAGE.inference / SAGEConv.forward_full), each bracketed by events
    parts = []
    for _ in range(3):
        rec = {}
        with torch.no_grad():
            holder = {}
            rec["rows"] = event_ms(lambda: holder.__setitem__("h", model._all_rows(n)))
            h = holder.pop("h")
            for l, layer in enumerate(model.layers):
                r = {}
                if layer.in_feats > layer.out_feats:
                    r["gemm_ms"] = event_ms(lambda: holder.__setitem__("t", layer.fc_neigh(h)))
                    r["agg_ms"] = event_ms(lambda: holder.__setitem__("a", gnn_ops.aggregate_full(g, holder["t"])))
                    r["agg_F"] = layer.out_feats
                else:
                    r["agg_ms"] = event_ms(lambda: holder.__setitem__("t", gnn_ops.aggregate_full(g, h)))
                    r["gemm_ms"] = event_ms(lambda: holder.__setitem__("a", layer.fc_neigh(holder["t"])))
                    r["agg_F"] = layer.in_feats
                a = holder.pop("a")
                holder.pop("t")

                def rest():
                    out = layer.fc_self(h)
                    out += a
                    out += layer.bias
                    if l != len(model.layers) - 1:
                        torch.relu_(out)
                    holder["h"] = out
                r["fc_self_bias_relu_ms"] = event_ms(rest)
                del a
                h = holder.pop("h")
                rec["layer%d" % l] = {k: (round(v, 3) if isinstance(v, float) else v) for k, v in r.items()}
            del h
        rec["rows"] = round(rec["rows"], 3)
        parts.append(rec)
    print(json.dumps({"gpu": gpu, "what": "SAGE.inference", "model": "SAGE(100, 256, 47, 3 layers), fbtt "
                      "(125, 140, 140) x (4, 5, 5), ranks 16, 16; dense layers: torch fp32 Linear",
                      "end_to_end": summary(ts), "peak_bytes_above_model_and_graph": peak,
                      "split_runs": parts}), flush=True)


if __name__ == "__main__":
    main()
