#!/usr/bin/env python
"""bench.py -- TT-EmbeddingBag fwd + bwd + fused SGD throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]

One step = one pass of the hot path over one batch of synthetic input at BASELINE config 2
("GraphSAGE on ogbn-products shape, FBTT p=125,140,140 q=4,5,5 ranks 16,16"): 262,144 distinct
uniformly drawn node ids (the size of a batch-1024, fanout [5,10,15] layer-0 frontier), one index
per bag, forward reconstruction of the rows, backward with an upstream gradient, fused SGD on the
cores.  Prints ONE JSON line (rank 0).

  value      rows/s with the inputs resident in HBM, the step replayed as a CUDA graph of the raw
             C-ABI ops (tt_forward + tt_sgd_backward); N > 1: each rank runs its own batch (weak
             scaling) and the dense core gradients are all-reduced over NCCL before the update
  e2e        the same metric through the module a user calls (TTEmbeddingBag.forward + autograd),
             indices / offsets copied from pinned host memory and the scalar loss read back every
             step
  roofline   dominant kernel, algorithmic bytes / CUDA-event duration vs the measured HBM peak
  cpu_baseline / --impl reference : the oracle's C port of the same step on the host cores, same rows per step
  sage / config3 / papers : sub-records of the same line -- the GraphSAGE epoch of BASELINE configs 2 and 3
             (bench_sage.sage_epoch_record: strong scaling over the N ranks, its own clock sample) and the
             TT step at the papers100M shape (config 5); `sage_epoch_s` repeats the config-2 epoch time at
             the top level.  --no-extra skips them.
  replicas_bit_identical (N > 1): checksums of the cores of all ranks after the timed steps

--dump-outputs DIR (rank 0): after the timed steps, what the last of them handed its caller, as float32 .npy files:
  tt_forward_rows.npy, a fixed seeded sample of up to 65,536 rows of the forward's output (sorted row positions
  drawn by numpy's default_rng(0); the whole output is 105 MB at the default batch), and core<t>.npy, the cores
  after that step's SGD update; 64 MB at most.  The inputs depend on the arguments only, so two builds can be
  compared file by file.

Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.
L2: four batches are rotated; one step touches 212 MB (> 126 MB L2), the rotation 850 MB.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _cublas_emulation  # noqa: E402,F401 -- before torch: the sub-records' dense GNN layers (see the module)

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "falcon-ttdforgnns_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

SHAPES = {
    "products": dict(n=2449029, p=[125, 140, 140], q=[4, 5, 5], ranks=[16, 16]),
    "arxiv": dict(n=169343, p=[55, 55, 56], q=[4, 4, 8], ranks=[16, 16]),
    "papers": dict(n=111059956, p=[481, 481, 481], q=[4, 4, 8], ranks=[32, 32]),
}
METRIC = "TT-EmbeddingBag rows/s fwd+bwd+SGD"
NUM_ROT = 4
LR = 0.01   # zero-mean upstream gradient + small step: the cores stay finite over any number of steps
DUMP_ROWS = 65536          # forward rows written by --dump-outputs
DUMP_MAX_BYTES = 64 << 20


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
                power.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "samples": len(sm),
                "power_w_max": max(power), "reasons": sorted(reasons)}


def dist_env():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return world, rank, local


# --------------------------------------------------------------------------------------------
# CPU baseline (oracle port) -- the only place bench.py executes oracle/
# --------------------------------------------------------------------------------------------
def cpu_step_rate(shape, sample_rows, steps, warmup, seed=0):
    from oracle import oracle as orc
    orc.use_all_host_threads()      # torchrun exports OMP_NUM_THREADS=1
    p, q, ranks = shape["p"], shape["q"], [1] + shape["ranks"] + [1]
    D = int(np.prod(q))
    rng = np.random.default_rng(seed)
    cores = [(rng.standard_normal((1, p[t], ranks[t] * q[t] * ranks[t + 1])) /
              np.sqrt(shape["n"])).astype(np.float32) for t in range(3)]
    cols = [ranks[t] * q[t] * ranks[t + 1] for t in range(3)]
    batches = [(rng.choice(shape["n"], size=sample_rows, replace=False).astype(np.int64),
                (rng.random((sample_rows, D)) * 0.1).astype(np.float32)) for _ in range(2)]

    def one(i):
        idx, d_out = batches[i % 2]
        orc.tt_forward_f32_rows(p, q, ranks, cores, idx)
        g = orc.tt_backward_f32_rows(p, q, ranks, cores, idx, d_out)
        orc.apply_optimizer(p, cols, "sgd", 0.1, 0.0, cores, None, g)

    for i in range(warmup):
        one(i)
    t0 = time.perf_counter()
    for i in range(steps):
        one(i)
    dt = time.perf_counter() - t0
    return sample_rows * steps / dt, dt / steps, orc.num_threads()


def calibrated_cpu_baseline(shape, target_seconds=12.0):
    rate, _, threads = cpu_step_rate(shape, 2048, 1, 1)
    rows = int(min(262144, max(2048, rate * target_seconds / 3)))
    rate, sec, threads = cpu_step_rate(shape, rows, 3, 1)
    return {"value": rate, "unit": "rows/s", "cores": threads, "kind": "port",
            "sample": "%d rows x 3 steps of the same workload (C oracle port, fp32, OpenMP), "
                      "%.2f s/step" % (rows, sec)}


def run_reference(args, shape):
    world, rank, _ = dist_env()
    if rank != 0:
        return
    rows = args.cpu_rows or min(args.nnz, shape["n"])      # same config as the GPU arm
    rate, sec, threads = cpu_step_rate(shape, rows, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(args), "rows_per_step": rows,
                   "note": "the reference has no CPU implementation of this path (CUDA only); "
                           "this is the oracle's C port of FBTT tt_forward + tt_sgd_backward on "
                           "all host threads, the same rows per step as the GPU arm; under torchrun "
                           "rank 0 alone runs it (one CPU job whatever N is)"},
        "cpu_baseline": {"value": rate, "unit": "rows/s", "cores": threads, "kind": "port",
                         "sample": "%d rows per step" % rows},
        "e2e": {"value": rate, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "reference_gpu": reference_gpu_rate(args, shape),
    }
    print(json.dumps(line), flush=True)


def reference_gpu_rate(args, shape, steps=5):
    """The reference's own CUDA kernels (oracle/_ref, built unmodified for sm_100a) on the full
    workload, device-resident inputs, CUDA events: reported beside the CPU number of the reference
    arm.  None when there is no GPU or the extension was not built."""
    try:
        from oracle import ref_ext
        rmod = ref_ext.load()
        if rmod is None or not torch.cuda.is_available():
            return None
        dev = torch.device("cuda", 0)
        p, q, rr, N = shape["p"], shape["q"], [1] + shape["ranks"] + [1], shape["n"]
        D, nnz = int(np.prod(q)), min(args.nnz, N)
        g = torch.Generator().manual_seed(1000)
        cores = [(torch.randn(1, p[t], rr[t] * q[t] * rr[t + 1], generator=g) / np.sqrt(N)).to(dev)
                 for t in range(3)]
        idx = [torch.randperm(N, generator=g)[:nnz].to(dev) for _ in range(NUM_ROT)]
        dout = [((torch.rand(1, nnz, D, generator=g) - 0.5) * 0.2).to(dev) for _ in range(NUM_ROT)]
        row = torch.arange(nnz, device=dev)
        tb = torch.zeros(nnz, dtype=torch.int64, device=dev)
        Lt = torch.tensor([p[1] * p[2], p[2], 1], dtype=torch.int64, device=dev)

        def one(k):
            rmod.tt_forward(1000, 1, nnz, D, p, q, rr, Lt, nnz, idx[k], row, tb, cores)
            rmod.tt_sgd_backward(1000, D, LR, p, q, rr, Lt, nnz, idx[k], row, tb, dout[k], cores)

        for i in range(2):
            one(i % NUM_ROT)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            one(i % NUM_ROT)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / steps
        return {"value": nnz / (ms * 1e-3), "unit": "rows/s", "ms_per_step": ms,
                "what": "reference FBTT tt_forward + tt_sgd_backward (batch_count 1000), unmodified "
                        "sources compiled for sm_100a, %d rows per step on one B200" % nnz}
    except Exception as ex:   # the CPU arm must not fail because the GPU extra did
        return {"unavailable": str(ex)[:200]}


def workload_name(args):
    s = SHAPES[args.shape]
    return ("%s shape: N=%d, p=%s q=%s ranks=%s, %d distinct uniform ids per step, one index per "
            "bag, fwd+bwd+SGD" % (args.shape, s["n"], s["p"], s["q"], s["ranks"], min(args.nnz, s["n"])))


# --------------------------------------------------------------------------------------------
# ours
# --------------------------------------------------------------------------------------------
class _DotLoss(torch.autograd.Function):
    """loss = <out, target>, the cheapest loss whose gradient (d_output = target) is arbitrary: one pass over
    `out` forward, and the backward hands `target` itself to the embedding (no multiply by the incoming 1.0:
    round 1 spent 98 us of a 331 us step in the benchmark's own loss arithmetic)."""

    @staticmethod
    def forward(ctx, out, target):
        ctx.target = target
        ctx.shape = out.shape
        return torch.dot(out.reshape(-1), target)

    @staticmethod
    def backward(ctx, grad):
        return ctx.target.view(ctx.shape), None


def tt_subrecord(shape_name, nnz, steps, warmup, world, rank, dev, exchange):
    """The same fwd + bwd + SGD step at another BASELINE shape (config 5: papers100M shape), raw C-ABI ops,
    eager launches, CUDA events, max over ranks; a sub-record of the JSON line."""
    import torch.distributed as dist
    import dp
    import tt_embeddings as te
    shape = SHAPES[shape_name]
    p, q, ranks, N = shape["p"], shape["q"], shape["ranks"], shape["n"]
    rr = [1] + ranks + [1]
    D = int(np.prod(q))
    nnz = min(nnz, N)
    g = torch.Generator().manual_seed(77)
    cores = [(torch.randn(1, p[t], rr[t] * q[t] * rr[t + 1], generator=g) / np.sqrt(N)).to(dev) for t in range(3)]
    g = torch.Generator().manual_seed(2000 + rank)
    # distinct ids over the whole range (ids beyond 2^24 and 2^31 / 4 at papers shape)
    idx = []
    for _ in range(2):
        u = torch.randint(0, N, (nnz + nnz // 8,), generator=g).unique()
        idx.append(u[torch.randperm(u.numel(), generator=g)][:nnz])       # distinct, unsorted
    nn = min(int(i.numel()) for i in idx)
    idx = [i[:nn].contiguous().to(dev) for i in idx]
    rowidx = torch.arange(nn, device=dev)
    tableidx = torch.zeros(nn, dtype=torch.int64, device=dev)
    d_out = [((torch.rand(1, nn, D, generator=g) - 0.5) * 0.2).to(dev) for _ in range(2)]
    xchg = None
    if world > 1 and exchange == "peer":
        try:
            xchg = dp.PeerExchange(cores)
        except Exception:
            xchg = None

    def step(k):
        te.tt_forward(1000, 1, nn, D, p, q, rr, None, nn, idx[k], rowidx, tableidx, cores)
        if world == 1:
            te.tt_sgd_backward(1000, D, LR, p, q, rr, None, nn, idx[k], rowidx, tableidx, d_out[k], cores)
        else:
            dc = te.tt_dense_backward(1000, D, p, q, rr, None, nn, idx[k], rowidx, tableidx, d_out[k], cores)
            if xchg is not None:
                xchg.step(dc, cores, "sgd", LR)
            else:
                dp.apply_optimizer(p, q, rr, cores, dp.allreduce_mean(dc), LR)

    for i in range(max(warmup, 3)):
        step(i % 2)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(i % 2)
    e1.record()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    failed = 0
    if xchg is not None:
        failed = xchg.failed_epoch()
        xchg.close()
    hbm_peak, _, _ = measured_peaks()
    step_bytes = nn * (16 + 8 * D) + 2 * sum(c.numel() * 4 for c in cores)
    return {"metric": METRIC, "value": world * nn / (ms * 1e-3), "unit": "rows/s", "ms_per_step": ms,
            "n_gpus": world, "steps": steps, "scaling": "weak", "launch": "eager",
            "workload": "%s shape: N=%d, p=%s q=%s ranks=%s, %d distinct ids per step and rank over the whole "
                        "index range" % (shape_name, N, p, q, ranks, nn),
            "step_frac_of_hbm_bound": (step_bytes / (hbm_peak * 1e9)) / (ms * 1e-3),
            "exchange_failed": failed}


def dump_outputs(out_dir, out, cores):
    """Writes the forward output `out` of one step (a fixed sample of its rows, as many as DUMP_MAX_BYTES leaves
    room for beside the cores) and the `cores` after that step's update to out_dir/<name>.npy (the --dump-outputs
    record, see the module docstring)."""
    arrays = {"core%d" % t: c.detach().float().cpu().numpy() for t, c in enumerate(cores)}
    out = out.reshape(-1, out.shape[-1])
    room = DUMP_MAX_BYTES - sum(a.nbytes for a in arrays.values())
    n = max(0, min(out.shape[0], DUMP_ROWS, room // (4 * out.shape[1])))
    rows = np.sort(np.random.default_rng(0).choice(out.shape[0], size=n, replace=False))
    arrays["tt_forward_rows"] = out[torch.from_numpy(rows).to(out.device)].float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def replicas_identical(tensors, dev):
    """All ranks hold bit-identical copies of `tensors`? (two checksums of the bit patterns, all-gathered)"""
    import torch.distributed as dist
    flat = torch.cat([t.detach().reshape(-1).view(torch.int32).to(torch.int64) for t in tensors])
    chk = torch.stack([flat.sum(), (flat * torch.arange(1, flat.numel() + 1, device=dev)).sum()])
    allc = [torch.empty_like(chk) for _ in range(dist.get_world_size())]
    dist.all_gather(allc, chk)
    return all(bool(torch.equal(allc[0], c)) for c in allc)


def run_ours(args, shape):
    import torch.distributed as dist
    world, rank, local = dist_env()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device (the product has no CPU path; "
                           "use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    json_out = sys.stdout
    if world > 1:
        # libraries write to file descriptor 1 (NCCL's version banner at NCCL_DEBUG=VERSION / WARN);
        # ours is ONE JSON line: keep a private copy of stdout for it and point fd 1 at stderr
        sys.stdout.flush()
        json_out = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    import _ttg
    import dp
    import pipeline
    import tt_embeddings as te
    from FBTT.tt_embeddings_ops import OptimType, TTEmbeddingBag

    lib = _ttg.lib()
    # The device-resident loop builds the next batch's plan on a stream forked at the START of the step (beside the
    # group table and the head of the forward): 172 vs 179 us per step.  Forked behind the forward, or with 8 SMs
    # left free (TTG_FLAG_SHARE_SMS), it gains nothing: a CTA of the row kernels takes a whole register file and
    # the dependent-launch CTAs of the next kernel take the spare SMs (profiles/r2_step_timeline.txt).
    # --no-plan-ahead restores the round-1 flow in both loops.
    share = 0
    te.EXTRA_FLAGS = int(args.flags) | share
    p, q, ranks, N = shape["p"], shape["q"], shape["ranks"], shape["n"]
    rr = [1] + ranks + [1]
    D = int(np.prod(q))
    nnz = min(args.nnz, N)     # distinct ids per step: a table smaller than the batch caps it
    torch.manual_seed(1234)
    module = TTEmbeddingBag(N, D, ranks, p, q, optimizer=OptimType.SGD, learning_rate=LR,
                            sparse=True, use_cache=False, weight_dist="normal")
    cores = [c.data for c in module.tt_cores]
    core_bytes = sum(c.numel() * 4 for c in cores)

    g = torch.Generator().manual_seed(1000 + rank)
    idx_host = [torch.randperm(N, generator=g)[:nnz].contiguous().pin_memory() for _ in range(NUM_ROT)]
    off_host = torch.arange(nnz + 1, dtype=torch.int64).pin_memory()
    idx_dev = [t.to(dev) for t in idx_host]
    rowidx = torch.arange(nnz, device=dev)
    tableidx = torch.zeros(nnz, dtype=torch.int64, device=dev)
    d_out = [((torch.rand(1, nnz, D, generator=g) - 0.5) * 0.2).to(dev) for _ in range(NUM_ROT)]
    groups = int(torch.unique(idx_host[0] // p[2]).numel())

    # N > 1: the exchange step is one kernel over NVLink peer memory (dp.PeerExchange); NCCL
    # all-reduce + optimizer launch only if the peers cannot be mapped (--exchange nccl forces it)
    xchg = None
    if world > 1 and args.exchange == "peer":
        try:
            xchg = dp.PeerExchange(cores)
        except Exception as ex:
            print("bench.py: peer exchange unavailable (%s); using the NCCL all-reduce" % ex,
                  file=sys.stderr)

    plan_stream = torch.cuda.Stream(dev)

    def plan_next(k):
        """the index plan of the NEXT batch, beside this step's kernels (it depends on the indices only): a fork
        of the current stream, joined at the end of the step; tt_forward finds it ready and skips its own"""
        if args.no_plan_ahead:
            return None
        cur = torch.cuda.current_stream(dev)
        plan_stream.wait_stream(cur)
        with torch.cuda.stream(plan_stream):
            kn = (k + 1) % NUM_ROT
            te.tt_plan(1, nnz, p, q, rr, nnz, idx_dev[kn], rowidx, tableidx, kn & 1)
        return cur

    def raw_step(k):
        cur = plan_next(k)
        out = te.tt_forward(1000, 1, nnz, D, p, q, rr, None, nnz, idx_dev[k], rowidx, tableidx, cores)
        raw_backward(k)
        if cur is not None:
            cur.wait_stream(plan_stream)
        return out

    def raw_backward(k):
        if world == 1:
            te.tt_sgd_backward(1000, D, LR, p, q, rr, None, nnz, idx_dev[k], rowidx, tableidx,
                               d_out[k], cores)
        else:
            dc = te.tt_dense_backward(1000, D, p, q, rr, None, nnz, idx_dev[k], rowidx, tableidx,
                                      d_out[k], cores)
            if xchg is not None:
                xchg.step(dc, cores, "sgd", LR)
            else:
                dp.apply_optimizer(p, q, rr, cores, dp.allreduce_mean(dc), LR)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # ---- warm-up (eager), then try to capture one CUDA graph per rotating batch
    NROT_W = ((max(args.warmup, 3) + NUM_ROT - 1) // NUM_ROT) * NUM_ROT    # whole rotations: batch k <-> slot k & 1
    for i in range(NROT_W):
        raw_step(i % NUM_ROT)
    sync_all()
    l0 = lib.ttg_launch_count()
    for k in range(NUM_ROT):
        raw_step(k)
    launches_per_step = int(lib.ttg_launch_count() - l0) // NUM_ROT
    sync_all()
    # with the NCCL all-reduce the step stays eager: capturing it works and is 8 % faster (0.2105
    # vs 0.2276 ms/step on 2 GPUs), but the process then hangs in destroy_process_group at exit
    # (measured once, 2026-10-18).  The peer-memory exchange is an ordinary kernel and captures.
    graphs, use_graph = [], ((world == 1 or xchg is not None) and not args.no_graph)
    graph_outs = []    # graph k's forward output, rewritten by every replay of graph k
    if use_graph:
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for k in range(NUM_ROT):
                    gr = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(gr, stream=side):
                        graph_outs.append(raw_step(k))
                    graphs.append(gr)
            torch.cuda.current_stream(dev).wait_stream(side)
            sync_all()
            for k in range(NUM_ROT):
                graphs[k].replay()
            sync_all()
        except Exception as ex:  # capture is an optimisation of the launch path, not a fallback
            print("bench.py: CUDA graph capture failed (%s); timing eager launches" % ex,
                  file=sys.stderr)
            graphs, use_graph = [], False
            sync_all()

    def timed(fn, steps):
        sync_all()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        sync_all()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    eager_out = [None]

    def eager_step(i):
        eager_out[0] = raw_step(i % NUM_ROT)

    step_fn = (lambda i: graphs[i % NUM_ROT].replay()) if use_graph else eager_step
    for i in range(((args.warmup + NUM_ROT - 1) // NUM_ROT) * NUM_ROT):
        step_fn(i)
    sampler = ClockSampler(local) if rank == 0 else None
    ms_total = timed(step_fn, args.steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:     # before any later step moves the cores on
        dump_outputs(args.dump_outputs, graph_outs[(args.steps - 1) % NUM_ROT] if use_graph else eager_out[0],
                     cores)
    ms_step = ms_total / args.steps
    value = world * nnz / (ms_step * 1e-3)

    # ---- per-kernel device time (eager, CUDA events inside the library)
    kern = {}
    if rank == 0 or world > 1:
        lib.ttg_profile_enable(1)
        nprof = min(args.steps, 20)
        for i in range(nprof):
            raw_step(i % NUM_ROT)
        torch.cuda.synchronize(dev)
        i = 0
        while lib.ttg_profile_name(i):
            tot, cnt = C.c_double(0), C.c_int64(0)
            lib.ttg_profile_read(i, C.byref(tot), C.byref(cnt))
            if cnt.value:
                kern[lib.ttg_profile_name(i).decode()] = {"ms": tot.value / cnt.value,
                                                          "launches_per_step": cnt.value / nprof}
            i += 1
        lib.ttg_profile_enable(0)

    # ---- the same step in the two other arithmetic modes (eager launches, CUDA events): context
    # for the headline number, not part of it
    alt_modes = None
    if world == 1 and not args.no_cpu_baseline and args.flags == 0:
        alt_modes = {}
        for name, fl in (("default_3xtf32", 0), ("tf32_single_pass", 8), ("fp32_ffma_kernels", 16)):
            te.EXTRA_FLAGS = fl | share
            for i in range(3):
                raw_step(i % NUM_ROT)
            ms_alt = timed(lambda i: raw_step(i % NUM_ROT), 10) / 10
            alt_modes[name] = {"ms_per_step_eager": ms_alt, "rows_per_s": nnz / (ms_alt * 1e-3)}
        te.EXTRA_FLAGS = int(args.flags) | share

    # ---- end to end through the module API (host indices in, scalar loss out).  Every step's
    # index arrays go pinned host -> device inside the timed region (on the copy stream of
    # pipeline.HostBatchPipeline, one step ahead of the kernels) and every step's loss comes back
    # to the host inside it (pipeline.DeferredScalars, read one step late; the last one is
    # drained before the closing event).  `e2e_sync` is the same loop with the copies on the
    # compute stream and loss.item() every step.
    # the loss is <out, target>: the cheapest one whose gradient (d_output = target) is arbitrary
    target = [d.view(-1) for d in d_out]
    module.sparse = (world == 1)   # N > 1: dense gradients, all-reduce, then the update

    def module_step(indices, offsets, k):
        out = module(indices, offsets)
        loss = _DotLoss.apply(out, target[k])
        loss.backward()
        if world > 1:  # data parallel: explicit exchange step instead of the fused update
            dp.dp_backward_step(module, [c.grad for c in module.tt_cores], exchange=xchg)
            for c in module.tt_cores:
                c.grad = None
        return loss

    # the module prepares a staged batch (bag -> row map, index plan) on the copy stream, beside the running step
    pipe = pipeline.HostBatchPipeline(
        dev, depth=2, on_staged=None if args.no_plan_ahead else (lambda slot, i, o: module.prepare(i, o, slot)))
    graphed = {}     # (staging slot, batch) -> the module step captured as a CUDA graph
    e2e_graph = use_graph   # with NCCL in the step it stays eager (see above)

    prof_e2e = os.environ.get("TTG_E2E_PROFILE") == "1"      # host time per call of the loop, to stderr
    host_t = {"get": 0.0, "put": 0.0, "step": 0.0, "release": 0.0, "push": 0.0}

    def e2e_pipelined(nsteps, use_graphs):
        reader = pipeline.DeferredScalars(dev, delay=1)
        got, h0 = [], pipe.h2d_bytes
        pipe.put(idx_host[0], off_host)
        clk = time.perf_counter
        for i in range(nsteps):
            k = i % NUM_ROT
            t0 = clk()
            indices, offsets = pipe.get()
            t1 = clk()
            if i + 1 < nsteps:
                pipe.put(idx_host[(i + 1) % NUM_ROT], off_host)
            t2 = clk()
            if use_graphs:
                gk = (indices.data_ptr(), k)
                gs = graphed.get(gk)
                if gs is None:   # warm-up only: NUM_ROT is a multiple of the pipeline depth
                    gs = graphed[gk] = pipeline.GraphedStep(
                        lambda: module_step(indices, offsets, k), dev)
                loss = gs()
            else:
                loss = module_step(indices, offsets, k)
            t3 = clk()
            pipe.release()
            t4 = clk()
            got += reader.push(loss)
            if prof_e2e:
                t5 = clk()
                for name, dt in (("get", t1 - t0), ("put", t2 - t1), ("step", t3 - t2), ("release", t4 - t3),
                                 ("push", t5 - t4)):
                    host_t[name] += dt
        if prof_e2e and nsteps > NUM_ROT:
            print("bench.py: e2e host us per step (graphs=%s): %s" %
                  (use_graphs, {n: round(v / nsteps * 1e6, 1) for n, v in host_t.items()}), file=sys.stderr)
        for n in host_t:
            host_t[n] = 0.0
        got += reader.drain()
        assert len(got) == nsteps
        return got, (pipe.h2d_bytes - h0) // nsteps, reader.d2h_bytes // nsteps

    idx_stage = torch.empty(nnz, dtype=torch.int64, device=dev)
    off_stage = torch.empty(nnz + 1, dtype=torch.int64, device=dev)

    def e2e_sync_step(i):
        k = i % NUM_ROT
        idx_stage.copy_(idx_host[k], non_blocking=True)
        off_stage.copy_(off_host, non_blocking=True)
        return float(module_step(idx_stage, off_stage, k).item())

    res = {}
    e2e_pipelined(NUM_ROT, False)
    e2e_eager_ms = timed(lambda i: res.update(r=e2e_pipelined(args.steps, False)), 1) / args.steps
    if e2e_graph:
        try:
            e2e_pipelined(NUM_ROT, True)      # captures the NUM_ROT graphs
            e2e_pipelined(NUM_ROT, True)
            n_before = len(graphed)
            e2e_ms = timed(lambda i: res.update(r=e2e_pipelined(args.steps, True)), 1) / args.steps
            assert len(graphed) == n_before, "a graph was captured inside the timed region"
        except Exception as ex:   # capture is an optimisation of the launch path, not a fallback
            print("bench.py: e2e graph capture failed (%s); reporting eager launches" % ex,
                  file=sys.stderr)
            e2e_graph = False
            sync_all()
            res.clear()
            e2e_eager_ms = timed(lambda i: res.update(r=e2e_pipelined(args.steps, False)), 1) / args.steps
    if not e2e_graph:
        e2e_ms = e2e_eager_ms
    losses, h2d_per_step, d2h_per_step = res["r"]
    e2e_value = world * nnz / (e2e_ms * 1e-3)
    for i in range(3):
        e2e_sync_step(i)
    e2e_sync_ms = timed(e2e_sync_step, args.steps) / args.steps

    exchange_failed, peer_exchange = 0, xchg is not None
    identical = None
    if world > 1:                 # every rank applied the same updates to the same cores?
        identical = replicas_identical(cores, dev)
    if xchg is not None:          # collective: before the ranks part ways
        exchange_failed = xchg.failed_epoch()
        xchg.close()
    # ---- the other BASELINE configs as sub-records (collective at N > 1: every rank runs them)
    extra = {}
    if not args.no_extra:
        import bench_sage
        mk = (lambda: ClockSampler(local)) if rank == 0 else None
        try:
            extra["papers"] = tt_subrecord("papers", args.nnz, min(args.steps, 20), 3, world, rank, dev,
                                           args.exchange)
        except Exception as ex:
            extra["papers"] = {"error": str(ex)[:300]}
            if world > 1:
                raise
        for name, cfg in (("sage", 2), ("config3", 3)):
            try:
                extra[name] = bench_sage.sage_epoch_record(world, rank, dev, config=cfg, epochs=args.sage_epochs,
                                                           flags=args.flags, clock_sampler=mk)
            except Exception as ex:   # a sub-record must not take the headline line down
                extra[name] = {"error": str(ex)[:300]}
                if world > 1:
                    raise
        # BASELINE config 4 (full-graph GCN / GAT at ogbn-arxiv shape) is a single-GPU recipe
        # (gcn_gat_partition.py): rank 0 runs it alone while the others wait at the end
        if rank == 0:
            try:
                import bench_fullgraph
                recs = bench_fullgraph.fullgraph_records(dev, epochs=5)
                extra["fullgraph"] = {r["metric"].split()[1].lower() + "_epoch_ms": r["value"] for r in recs}
                extra["fullgraph"]["records"] = recs
            except Exception as ex:
                extra["fullgraph"] = {"error": str(ex)[:300]}
        if world > 1:
            dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if exchange_failed:
        print("bench.py: a peer did not arrive at exchange step %d; the numbers are invalid"
              % exchange_failed, file=sys.stderr)

    # ---- roofline
    hbm_peak, peak_src, sm_max = measured_peaks()
    bytes_fwd = nnz * (8 + 4 * D)
    bytes_bwd = nnz * (8 + 4 * D)
    alg = {"fwd_rows_kernel": bytes_fwd, "bwd_rows_kernel": bytes_bwd,
           "generic_fwd_kernel": bytes_fwd, "generic_bwd_kernel": bytes_bwd}
    dom = max((k for k in kern if k in alg), key=lambda k: kern[k]["ms"], default=None)
    # DRAM traffic per launch of the dominant kernel: from the committed ncu capture of this round
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "kernel_traffic.json")
    if dom and os.path.exists(tpath) and args.shape == "products" and nnz == 262144:
        t = json.load(open(tpath)).get(dom)
        if t:
            traffic, traffic_src = t["dram_bytes_per_launch"], t["source"]
    roofline = None
    if dom:
        achieved = alg[dom] / (kern[dom]["ms"] * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm_peak,
                    "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                    "traffic_source": traffic_src, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": alg[dom], "kernel_ms": kern[dom]["ms"]}
    step_bytes = nnz * (16 + 8 * D) + 2 * core_bytes
    q0, q1, q2 = q
    r1, r2 = ranks
    f_row = 2 * (q0 * q1) * r2 * q2 * 3            # per row: row product, d_core2 slice, d(tr0)
    f_grp = 2 * q0 * r1 * (q1 * r2) * 4            # per group: tr0 fwd, tr0 bwd, d_core1, d_core0
    step_flops = f_row * nnz + f_grp * groups
    # pipe ceilings measured on this pool's B200 (profiles/r1_pipe_peaks.txt): fp32 FFMA with
    # three register operands 47 TFLOP/s, mma.sync TF32 m16n8k8 278 TFLOP/s
    ffma_peak, tf32_peak = 47.0e12, 278.0e12
    passes = 1 if (args.flags & 8) else 3          # 3xTF32 issues three tensor-core passes
    uses_tensor = not (args.flags & 16)
    t_hbm = step_bytes / (hbm_peak * 1e9)
    t_pipe = step_flops * passes / tf32_peak if uses_tensor else step_flops / ffma_peak
    bound_s = max(t_hbm, t_pipe)
    step_roofline = {
        "bytes_per_step": step_bytes, "flops_per_step_with_prefix_reuse": step_flops,
        "unique_groups": groups, "t_hbm_us": t_hbm * 1e6, "t_pipe_us": t_pipe * 1e6,
        "pipe": ("mma.sync tf32 x%d passes @ 278 TFLOP/s measured" % passes) if uses_tensor
                else "fp32 ffma @ 47 TFLOP/s measured",
        "bound": "pipe" if t_pipe > t_hbm else "hbm",
        "frac_of_bound": bound_s / (ms_step * 1e-3),
        "flops_per_step_no_reuse": nnz * (2 * q0 * r1 * q1 * r2 * 4 + 2 * q0 * q1 * r2 * q2 * 3),
    }
    kernel_share = {k: v["ms"] * v["launches_per_step"] for k, v in kern.items()}
    tot_k = sum(kernel_share.values()) or 1.0
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = calibrated_cpu_baseline(shape)
    # the reference's own CUDA kernels (unmodified, built for sm_100a by oracle/build_ref.py) on
    # the same batches: a GPU baseline beside the CPU one; absent when oracle/_ref was not built
    ref_gpu = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import ref_ext
        rmod = ref_ext.load()
        if rmod is not None:
            Lt = torch.tensor([p[1] * p[2], p[2], 1], dtype=torch.int64, device=dev)
            rcores = [c.clone() for c in cores]

            def ref_step(i):
                k = i % NUM_ROT
                rmod.tt_forward(1000, 1, nnz, D, p, q, rr, Lt, nnz, idx_dev[k], rowidx, tableidx, rcores)
                rmod.tt_sgd_backward(1000, D, LR, p, q, rr, Lt, nnz, idx_dev[k], rowidx, tableidx,
                                     d_out[k], rcores)

            for i in range(2):
                ref_step(i)
            rms = timed(ref_step, 5) / 5
            ref_gpu = {"value": nnz / (rms * 1e-3), "unit": "rows/s", "ms_per_step": rms,
                       "what": "reference FBTT tt_forward + tt_sgd_backward (batch_count 1000), "
                               "unmodified sources compiled for sm_100a, same batches, CUDA events"}
    line = {
        "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "rows_per_step_per_gpu": nnz,
                   "arithmetic": ("plain TF32 tensor-core passes (TTG_FLAG_TF32)" if (args.flags & 8)
                                  else "fp32 FFMA kernels (TTG_FLAG_FFMA)" if (args.flags & 16)
                                  else "fp32 via 3xTF32 split on tensor cores, fp32 accumulation"),
                   "l2": "4 rotating batches, 212 MB touched per step (> 126 MB L2)",
                   "launch": "cuda_graph" if use_graph else "eager",
                   "index_plan": "inside the forward" if args.no_plan_ahead else
                                 "of batch i + 1 built beside step i on a forked stream (ttg_tt_plan, second plan slot)",
                   "parallelism": "dp%d, replicated cores%s" % (
                       world, "" if world == 1 else
                       ", d_cores exchanged and the update applied by one kernel over NVLink peer memory"
                       if peer_exchange else ", NCCL all-reduce of d_cores per step")},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "rows/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(h2d_per_step), "d2h_bytes_per_step": int(d2h_per_step),
                "api": "TTEmbeddingBag.forward(indices, offsets), loss = dot(out, target) (backward hands target over as d_output), loss.backward(); indices and "
                       "offsets staged from pinned host memory one step ahead on a copy stream "
                       "(pipeline.HostBatchPipeline), the loss read back every step, one step "
                       "late (pipeline.DeferredScalars)" + (
                           "; the module step replayed as a CUDA graph (pipeline.GraphedStep)"
                           if e2e_graph else ""),
                "launch": "cuda_graph" if e2e_graph else "eager",
                "index_plan": "inside the forward" if args.no_plan_ahead else
                              "TTEmbeddingBag.prepare on the copy stream right behind the batch's host-to-device copy",
                "ms_per_step_eager_pipelined": e2e_eager_ms,
                "ms_per_step_eager_unpipelined": e2e_sync_ms,
                "loss_last": losses[-1] if losses else None},
        "gpu_launches": launches_per_step * args.steps,
        "gpu_launches_per_step": launches_per_step,
        "roofline": roofline,
        "step_roofline": step_roofline,
        "kernels_ms": {k: round(v["ms"], 5) for k, v in kern.items()},
        "kernel_share": {k: round(v / tot_k, 4) for k, v in kernel_share.items()},
        "cpu_baseline": cpu,
        "reference_gpu": ref_gpu,
        "alt_modes": alt_modes,
        "replicas_bit_identical": identical,
        "exchange_failed": exchange_failed,
        "sage_epoch_s": (extra.get("sage") or {}).get("value"),
        "sage": extra.get("sage"),
        "config3": extra.get("config3"),
        "papers": extra.get("papers"),
        "fullgraph": extra.get("fullgraph"),
        # the sub-records' dense GNN layers (torch library GEMMs, not the TT path): which cuBLAS ran them
        "library_gemms": ("fp32 on " + _cublas_emulation.WHY) if _cublas_emulation.ACTIVE
                         else "fp32 on torch's bundled cuBLAS (%s)" % _cublas_emulation.WHY,
    }
    print(json.dumps(line), file=json_out, flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default="products", choices=sorted(SHAPES))
    ap.add_argument("--nnz", type=int, default=262144)
    ap.add_argument("--cpu-rows", type=int, default=0,
                    help="rows per step of the --impl reference (CPU) arm; 0 = the same rows per step as "
                         "the GPU arm (--nnz)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: how the core gradients are exchanged")
    ap.add_argument("--flags", type=int, default=0,
                    help="TTG_FLAG_* bits OR-ed into every tt_forward / tt_backward call "
                         "(8 = plain TF32 tensor-core mode, 16 = fp32 FFMA kernels)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-plan-ahead", action="store_true",
                    help="build every batch's index plan inside its own forward (round-1 behaviour) instead of "
                         "beside the running step (forked stream / copy stream)")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the sub-records (GraphSAGE epoch of configs 2 and 3, papers-shape step)")
    ap.add_argument("--sage-epochs", type=int, default=5, help="timed GraphSAGE epochs per sub-record (the best one counts)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU step of --impl ours")
    if args.warmup < 3:
        args.warmup = 3
    shape = SHAPES[args.shape]
    if args.impl == "reference":
        run_reference(args, shape)
    else:
        run_ours(args, shape)


if __name__ == "__main__":
    main()
