#!/usr/bin/env python
"""bench.py — graphs/sec through the message-passing hot path, forward + backward (BASELINE.json metric).

    python bench.py [--config NAME] [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

--config picks the BASELINE.json configuration (default `masking`, the one the metric is quoted on):

    masking         configs[1]  chem/pretrain_masking.py:46-70     5-layer GIN-300, B = 256, Linear(300,119) + CE(fp64)
    contextpred     configs[2]  chem/pretrain_contextpred.py:50-97 5-layer + 3-layer GIN, B = 128 pairs, BCE(fp64)
    bio_supervised  configs[3]  bio/pretrain_supervised.py:25-42   bio GIN GNN_graphpred, B = 64 per GPU, T = 5000, BCE(fp64)
    gcn|gat|graphsage configs[4] the masking step with gnn_type swapped, B = 256

A step is the script's train() body between `batch.to(device)` and `optimizer.step()` (pretrain-gnns_b200/train_steps.py);
optimizer steps are excluded (SURVEY.md 8(d)).  With N > 1 every rank draws its own batches (weak scaling, graphs sharded by
rank) and the step includes ONE all-reduce of the gradients.

One JSON line is printed by rank 0.  `value` times K steps with the batches already resident in HBM (graph bucketing
included: every step sees a different batch).  `e2e` times the same K steps from pinned host memory: one packed pinned
buffer and one asynchronous H2D copy per step inside the timed region (the next batch prefetched under the running step) and
one D2H read of the loss per step (issued asynchronously after the step, consumed two steps later, as the reference's
`loss_accum += loss.item()` only feeds a log line).  L2 is flushed between timed steps (256 MiB memset outside the per-step
event pairs).  `--impl reference` times the reference's OWN model.py on the host cores (oracle/reference_runner.py;
kind "reference"), or the oracle port of it when the reference's sources are not on the box (kind "port").

`--dump-outputs DIR` writes, after the timed steps, what the last timed step on the resident batches handed its caller:
DIR/loss.npy (float64) and DIR/grad.<parameter>.npy (float32) for every parameter.  Batches and initial parameters are
seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import gc
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NUM_LAYER, EMB = 5, 300
NUM_DISTINCT_BATCHES = 8
METRIC = "graphs/sec 5-layer GIN-300 fwd+bwd on ZINC-shaped batches"
CONFIG_NAMES = ("masking", "contextpred", "bio_supervised", "gcn", "gat", "graphsage")
WORKLOADS = {
    "masking": "chem pretrain_masking 5-layer GIN emb_dim=300 batch_size=256 (BASELINE configs[1])",
    "contextpred": "chem pretrain_contextpred 5-layer GIN emb_dim=300 batch_size=128, substruct + 3-layer context encoders (BASELINE configs[2])",
    "bio_supervised": "bio pretrain_supervised 5-layer GIN emb_dim=300 PPI-ego-shaped graphs (~500 nodes) batch_size=64 per GPU, T=5000 (BASELINE configs[3])",
    "gcn": "chem pretrain_masking gnn_type=gcn emb_dim=300 batch_size=256 (BASELINE configs[4])",
    "gat": "chem pretrain_masking gnn_type=gat emb_dim=300 batch_size=256 (BASELINE configs[4])",
    "graphsage": "chem pretrain_masking gnn_type=graphsage emb_dim=300 batch_size=256 (BASELINE configs[4])",
}
PER_GPU_BATCH = {"masking": 256, "contextpred": 128, "bio_supervised": 64, "gcn": 256, "gat": 256, "graphsage": 256}


def metric_name(config):
    return METRIC if config == "masking" else "graphs/sec fwd+bwd, %s" % config


def base_config(config, world):
    """The `config` object of the JSON line: the SAME keys and values from both arms (arm-specific facts go to `detail`)."""
    B = PER_GPU_BATCH[config]
    return {"workload": WORKLOADS[config], "name": config, "global_batch": B * world, "per_gpu_batch": B, "parallelism": "dp%d" % world,
            "optimizer_step": "excluded (SURVEY 8(d))", "l2": "flushed between timed steps (256 MiB memset) on the GPU arm"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor=d["bf16_tflops"], tensor_sustained=d.get("bf16_tflops_sustained"), src="measured")
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, src="fallback")


def measured_traffic():
    """DRAM bytes per launch of the two roofline kernels from this round's `ncu --set full` captures: profiles/traffic.json,
    written by tools/ncu_traffic.py from the committed capture (never a constant typed into this file)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


class ClockSampler:
    """SM clock / throttle reasons sampled every 50 ms while the timed region runs.

    In-process NVML (nvidia_ml_py) in a daemon thread: spawning `nvidia-smi -lms` next to the timed region made the
    first end-to-end measurement on a fresh box ~2x slower (its start-up contends for the driver while the step is
    CPU-launch-bound); nvidia-smi is only the fallback when NVML cannot be imported."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.stop = index, [], None, False
        self.sm, self.mx, self.reasons, self.t = [], [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
        except Exception:
            self.nv = None

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[i])
            except Exception:
                return i
        return i

    def _poll(self):
        nv = self.nv
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        # the maximum clock is a constant of the board and nvmlDeviceGetMaxClockInfo is the one slow call here (1.5-19 ms measured,
        # tools/diag_nvml.py, against 3-8 us for the other two): query it once, before the timed region
        try:
            self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)))
        except Exception:
            pass
        while not self.stop:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def __enter__(self):
        if os.environ.get("PGNN_BENCH_NO_CLOCKS") == "1":   # diagnostic: no sampler thread at all (the line then carries no clocks)
            return self
        if self.nv is not None:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            try:
                self.sm.append(float(r[1])); self.mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:
                pass

    def __exit__(self, *a):
        self.stop = True
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
        if self.t is not None:
            self.t.join(timeout=2)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(self.mx), "reasons": sorted(self.reasons), "samples": len(sm),
                "source": "nvml" if self.nv is not None else "nvidia-smi"}


def dist_stats(xs):
    s = sorted(xs)
    n = len(s)
    return {"mean": sum(s) / n, "median": s[n // 2], "p95": s[min(n - 1, int(0.95 * n))], "max": s[-1], "min": s[0]}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the reference's own model.py (or the oracle port of it) on the host cores
# ---------------------------------------------------------------------------------------------------
def cpu_run(config, steps, warmup, batches=None, one_thread=False, threads=None):
    from oracle import reference_runner as R
    from oracle import steps_oracle as S
    ts = importlib.import_module("pretrain-gnns_b200.train_steps")
    cores = os.cpu_count() or 1
    B = PER_GPU_BATCH[config]
    P = S.make_params(config, 1, randomize_bn=False)
    if R.available():
        kind = "reference"
        step = S.REFERENCE_STEPS[config]()
        step.load(P)
        what = "the reference's own %s/model.py over the PyG-1.0.3 stand-in" % ("bio" if config == "bio_supervised" else "chem")
    else:
        kind = "port"
        step = S.PortStep(config, P)
        what = "the oracle port of the reference's model.py (its sources are not on this box)"
    batches = batches or ts.make_batches(config, 0, 2)
    heavy = config == "bio_supervised"   # seconds per step: keep the sample bounded

    def run(b):
        return float(step(b).detach())

    if threads is None:
        # "all the host threads it can use": these ops are small, so past a point more threads only add synchronisation
        # cost (128 threads: 25 graphs/s, measured); probe powers of two and keep the fastest (median of 3 after a warm-up)
        cand = sorted({c for c in ((16, 32) if heavy else (4, 8, 16, 32, 64)) if c <= cores} | {min(cores, 8)})
        best = (float("inf"), 1)
        for c in cand:
            torch.set_num_threads(c)
            run(batches[0])
            ts_ = []
            for _ in range(1 if heavy else 3):
                t0 = time.perf_counter()
                run(batches[0])
                ts_.append(time.perf_counter() - t0)
            best = min(best, (sorted(ts_)[len(ts_) // 2], c))
        threads = best[1]
    torch.set_num_threads(threads)
    for i in range(warmup):
        run(batches[i % len(batches)])
    per = []
    for i in range(steps):
        t0 = time.perf_counter()
        run(batches[i % len(batches)])
        per.append(time.perf_counter() - t0)
    total = sum(per)
    one = None
    if one_thread and not heavy:  # SURVEY.md 8(d): "also report a 1-thread figure"
        torch.set_num_threads(1)
        run(batches[0])
        t0 = time.perf_counter()
        for i in range(2):
            run(batches[i % len(batches)])
        one = B * 2 / (time.perf_counter() - t0)
        torch.set_num_threads(threads)
    return dict(value=B * steps / total, ms_per_step=1e3 * total / steps, cores=threads, value_1thread=one, kind=kind,
                per_step_ms=dist_stats([1e3 * t for t in per]),
                sample="%d fwd+bwd steps (after %d warm-up) of the B=%d %s batch: %s, torch CPU, best of the probed thread counts = %d of %d "
                       "host cores" % (steps, warmup, B, config, what, threads, cores))


def run_reference(args, rank):
    if rank != 0:
        return
    heavy = args.config == "bio_supervised"
    warmup = min(args.warmup, 1 if heavy else 5)
    r = cpu_run(args.config, args.steps, warmup)
    line = {"impl": "reference", "metric": metric_name(args.config), "value": r["value"], "unit": "graphs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": base_config(args.config, args.gpus),
            "detail": {"steps_timed": args.steps, "warmup_run": warmup, "per_step_ms": r["per_step_ms"],
                       "note": "host cores only; rank 0 runs one replica whatever --gpus says (the reference has no data parallelism)"},
            "cpu_baseline": {"value": r["value"], "unit": "graphs/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# analytic work per step (SURVEY.md 8(d)): GEMM flops and gather bytes from the batch's own sizes
# ---------------------------------------------------------------------------------------------------
def work_model(config, b):
    D = EMB
    if config == "contextpred":
        encs = [(5, int(b["x_substruct"].shape[0]), int(b["edge_index_substruct"].shape[1])), (3, int(b["x_context"].shape[0]), int(b["edge_index_context"].shape[1]))]
        head_flops = 0.0
        n, e = encs[0][1], encs[0][2]
        per_node = 2.0 * (D * 2 * D + 2 * D * D)
        gather = ("k_aggregate_fwd", 4 * D * (e + 2 * n))
        top = (n, 2 * D, D)
    elif config == "bio_supervised":
        n, e = int(b["x"].shape[0]), int(b["edge_index"].shape[1])
        encs = [(5, n, e)]
        per_node = 2.0 * (2 * D * 2 * D + 2 * D * D)
        T = int(b["go_target_pretrain"].numel() // b["center_node_idx"].shape[0])
        head_flops = 3 * 2.0 * b["center_node_idx"].shape[0] * 2 * D * T
        gather = ("k_aggregate_fwd", 4 * D * (e + n) + 4 * 2 * D * n)   # rows read (E+N) x D, rows written N x 2D (concat form)
        top = (n, 2 * D, 2 * D)
    else:
        n, e = int(b["x"].shape[0]), int(b["edge_index"].shape[1])
        encs = [(5, n, e)]
        m = int(b["masked_atom_indices"].shape[0])
        head_flops = 3 * 2.0 * m * D * 119
        if config == "masking":
            per_node, top = 2.0 * (D * 2 * D + 2 * D * D), (n, 2 * D, D)
            gather = ("k_aggregate_fwd", 4 * D * (e + 2 * n))
        elif config == "gat":
            per_node, top = 2.0 * D * 2 * D, (n, 2 * D, D)
            gather = ("k_gat_fwd", 4 * 2 * D * (e + n) + 4 * D * n)       # [N, heads*D] rows read per message, [N, D] written
        else:
            per_node, top = 2.0 * D * D, (n, D, D)
            gather = ("k_aggregate_fwd", 4 * D * (e + 2 * n))
    flops = head_flops + sum(3.0 * L * nn * per_node for L, nn, _ in encs)   # fwd + dgrad + wgrad
    return dict(gemm_flops_per_step=flops, gather_kernel=gather[0], gather_bytes_per_launch=gather[1], top_gemm=top,
                nodes=sum(nn for _, nn, _ in encs), edges=sum(ee for _, _, ee in encs))


# ---------------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist
    ts = importlib.import_module("pretrain-gnns_b200.train_steps")
    ops = importlib.import_module("pretrain-gnns_b200.ops")
    cabi = importlib.import_module("pretrain-gnns_b200._cabi")
    pdist = importlib.import_module("pretrain-gnns_b200.dist")
    pdata = importlib.import_module("pretrain-gnns_b200.data")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: there is no CPU fallback (use --impl reference)")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if args.precision:
        ops.set_precision(args.precision)
    torch.manual_seed(0)
    config = args.config
    B = PER_GPU_BATCH[config]
    step = ts.CONFIGS[config](dev)
    params = step.parameters()
    reducer = None
    if world > 1:
        srcs = [pdist.encoder_flat_source(m) for m in step.flat_sources() if hasattr(m, "_fused_plan")]
        reducer = pdist.GradAllReducer(params, flat_sources=srcs)

    host = step.make_batches(rank, NUM_DISTINCT_BATCHES)
    resident = [{k: v.to(dev) for k, v in b.items()} for b in host]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def train_step(b):
        loss = step(b)
        if reducer is not None:
            reducer.all_reduce_mean()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # end to end: every batch is ONE pinned buffer and ONE asynchronous copy on a side stream (data.BatchStager); the copy of
    # batch i+1 is issued right after step i has been enqueued, so it runs under step i's kernels.  Each of the K timed steps
    # contains exactly one host->device copy and one device->host read of its loss: the 8-byte copy into pinned memory is
    # enqueued behind the step and its value is consumed while the NEXT step runs (the reference only accumulates it for a log
    # line, chem/pretrain_masking.py:76), so the host never idles the GPU; the last read is inside the timed region too.
    stager = pdata.BatchStager(dev)
    packed = [stager.pack(b) for b in host]
    h2d_bytes = packed[0].nbytes
    LAG = 2  # the loss of step i is consumed while step i + LAG runs: the host may run up to LAG steps ahead of the GPU
    loss_host = torch.zeros(LAG + 1, dtype=torch.float64).pin_memory()
    loss_ready = [torch.cuda.Event() for _ in range(LAG + 1)]

    def timed(e2e):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        barrier()  # ranks finish their (CPU-side) setup seconds apart; start the first exchange together
        for i in range(args.warmup):
            b = stager.take(stager.submit(packed[i % len(packed)])) if e2e else resident[i % len(resident)]
            train_step(b).item()
        barrier()
        n0 = cabi.lib.pgnn_kernel_launch_count()
        gc.collect()
        gc.disable()  # a collection in the middle of the loop stalls the launch thread for milliseconds (seen as 2-9 ms steps)
        t0 = time.perf_counter()
        ticket, acc = None, 0.0
        host_t = []
        prof_step = int(os.environ.get("PGNN_BENCH_PROFILE_STEP", "-1")) if e2e else -1   # diagnostic: cProfile ONE iteration
        for i in range(args.steps):
            host_t.append(time.perf_counter())
            if i == prof_step:
                import cProfile
                pr = cProfile.Profile(); pr.enable()
            elif i == prof_step + 1 and prof_step >= 0:
                import io, pstats
                pr.disable(); buf = io.StringIO(); pstats.Stats(pr, stream=buf).sort_stats("tottime").print_stats(12)
                print(buf.getvalue(), file=sys.stderr, flush=True)
            flush.zero_()  # L2 flush, outside the per-step event pair
            ev[i][0].record()
            if e2e:
                if ticket is None:
                    ticket = stager.submit(packed[i % len(packed)])
                loss = train_step(stager.take(ticket))
                ticket = stager.submit(packed[(i + 1) % len(packed)]) if i + 1 < args.steps else None
                slot = i % (LAG + 1)
                loss_host[slot].copy_(loss.detach(), non_blocking=True)   # D2H read of this step's loss
                loss_ready[slot].record()
                if i >= LAG:  # consume an earlier step's loss while this one runs
                    j = (i - LAG) % (LAG + 1)
                    loss_ready[j].synchronize()
                    acc += float(loss_host[j])
            else:
                loss = train_step(resident[i % len(resident)])
            ev[i][1].record()
        if e2e:
            for i in range(max(args.steps - LAG, 0), args.steps):
                j = i % (LAG + 1)
                loss_ready[j].synchronize()
                acc += float(loss_host[j])
        barrier()
        wall = time.perf_counter() - t0
        gc.enable()
        launches = cabi.lib.pgnn_kernel_launch_count() - n0
        per = [a.elapsed_time(b) for a, b in ev]
        host_t.append(t0 + wall)
        timed.host_issue_ms = [1e3 * (b - a) for a, b in zip(host_t[:-1], host_t[1:])]  # host time per loop iteration (diagnostic)
        t = torch.tensor([sum(per)], dtype=torch.float64, device=dev)
        if world > 1:
            # every rank's own figures (sum, slowest step and its index), so that a slow rank can be told from a slow step
            mine = torch.tensor([sum(per), max(per), float(per.index(max(per))), sorted(per)[len(per) // 2]], dtype=torch.float64, device=dev)
            allr = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allr, mine)
            timed.per_rank = [dict(rank=r, ms_per_step=float(v[0]) / max(args.steps, 1), median_ms=float(v[3]), slowest_ms=float(v[1]),
                                   slowest_step=int(v[2])) for r, v in enumerate(allr)]
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        else:
            timed.per_rank = None
        timed.last_loss = loss if args.steps else None
        return float(t.item()), launches, wall, per, acc / max(args.steps, 1)

    with ClockSampler(local_rank) as clocks:
        ms_dev, launches, wall_dev, per_dev, _ = timed(False)
        # copied before the end-to-end pass below recomputes (and so overwrites) the gradients
        outputs = step_outputs(step, timed.last_loss) if args.dump_outputs and rank == 0 else None
        host_dev = timed.host_issue_ms
        per_rank_dev = timed.per_rank
        ms_e2e, _, wall_e2e, per_e2e, mean_loss = timed(True)
        host_e2e = timed.host_issue_ms
        per_rank_e2e = timed.per_rank
    graphs = B * world * args.steps
    wm = work_model(config, host[0])

    roof = roof_gather = None
    if rank == 0:
        roof, roof_gather = kernel_rooflines(ops, config, resident[0], dev, wm)
        if world == 1:
            try:  # per-kernel durations INSIDE the step (library timing mode: CUDA event pairs around every launch, warm L2)
                in_step_rooflines(cabi, train_step, resident, flush, roof, roof_gather, wm)
            except Exception as e:  # diagnostic only: the isolated timings above stand
                print("[bench] in-step kernel timing skipped: %s: %s" % (type(e).__name__, e), file=sys.stderr, flush=True)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:  # N=1 only
        heavy = config == "bio_supervised"
        cpu = cpu_run(config, 3 if heavy else 10, 1 if heavy else 3, batches=host[:2], one_thread=True)
    if rank != 0:
        return
    cfg = base_config(config, world)
    line = {
        "metric": metric_name(config), "value": graphs / (ms_dev * 1e-3), "unit": "graphs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32" if ops.get_precision() == "fp32" else "tf32x3", "data": "synthetic",
        "config": cfg,
        "detail": {"nodes_per_batch": wm["nodes"], "edges_per_batch": wm["edges"], "distinct_batches": NUM_DISTINCT_BATCHES,
                   "gemm_precision": ops.get_precision() + (" (error-compensated 3xTF32 on tcgen05, fp32-class: measured 1-3e-6 of scale; "
                                                            "--precision fp32 runs the exact FFMA kernels)" if ops.get_precision() != "fp32" else ""),
                   "grad_allreduce": (reducer.backend if reducer is not None else "none (1 GPU)"),
                   "per_step_ms": dist_stats(per_dev), "per_step_ms_e2e": dist_stats(per_e2e),
                   "slowest_steps": [(round(t, 3), i, round(host_dev[i], 3)) for t, i in sorted(((t, i) for i, t in enumerate(per_dev)), reverse=True)[:4]],
                   "slowest_e2e_steps": [(round(t, 3), i, round(host_e2e[i], 3)) for t, i in sorted(((t, i) for i, t in enumerate(per_e2e)), reverse=True)[:4]],
                   "slowest_steps_fields": "[device ms, step index, host ms spent issuing that loop iteration]",
                   "per_rank": per_rank_dev, "per_rank_e2e": per_rank_e2e,
                   "wall_ms_per_step_incl_flush": 1e3 * wall_dev / args.steps, "wall_ms_per_step_incl_flush_e2e": 1e3 * wall_e2e / args.steps,
                   "mean_loss_e2e": mean_loss, "gemm_flops_per_step": wm["gemm_flops_per_step"]},
        "e2e": {"value": graphs / (ms_e2e * 1e-3), "unit": "graphs/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 8,
                "ms_per_step": ms_e2e / args.steps,
                "transport": "one pinned buffer + one async H2D copy per batch on a side stream, next batch prefetched under the step "
                             "(data.BatchStager); loss copied to pinned memory after every step and consumed two steps later"},
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "roofline": roof, "roofline_gather": roof_gather,
        "cpu_baseline": None if cpu is None else {"value": cpu["value"], "unit": "graphs/s", "cores": cpu["cores"], "kind": cpu["kind"],
                                                  "sample": cpu["sample"], "value_1thread": cpu["value_1thread"]},
    }
    print(json.dumps(line), flush=True)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)


def step_outputs(step, loss):
    """What a training step hands its caller: the loss and every parameter's gradient, copied to host memory."""
    if loss is None:
        raise SystemExit("--dump-outputs needs at least one timed step")
    out = {"loss": loss.detach().double().cpu().numpy()}
    for name, p in step.named_parameters():
        if p.grad is not None:
            out["grad." + name] = p.grad.detach().float().cpu().numpy()
    return out


def dump_outputs(directory, outputs, limit=64 << 20):
    total = sum(a.nbytes for a in outputs.values())
    if total > limit:
        raise SystemExit("--dump-outputs: %d bytes of outputs exceed the %d-byte limit" % (total, limit))
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def _profile_rows(cabi, fn, steps):
    import ctypes
    lib = cabi.lib
    torch.cuda.synchronize()
    lib.pgnn_profile_read(None, 0)  # drop anything recorded earlier
    lib.pgnn_profile_enable(1)
    try:
        for i in range(steps):
            fn(i)
        torch.cuda.synchronize()
    finally:
        lib.pgnn_profile_enable(0)
    buf = ctypes.create_string_buffer(1 << 16)
    n = lib.pgnn_profile_read(buf, len(buf))
    rows = {}
    for line in buf.value.decode(errors="replace").splitlines():
        name, cnt, us = line.rsplit("\t", 2)
        rows[name] = (int(cnt), float(us))
    if n <= 0 or not rows:
        raise RuntimeError("no launches recorded")
    return rows


def _short(nm):  # "_ZN..17k_gemm_3xtf32_tmaILb0ELb0ELi224ELb0EEEv..." -> "k_gemm_3xtf32_tma<0,0,224,0>"
    import re
    m = re.search(r"(k_[A-Za-z0-9_]+?)(I(?:L[bi]\d+E)+E)?(?:Ev|E?P|$)", nm)
    if not m:
        return nm[:60]
    targs = re.findall(r"L[bi](\d+)E", m.group(2) or "")
    return m.group(1) + ("<" + ",".join(targs) + ">" if targs else "")


def in_step_rooflines(cabi, train_step, resident, flush, roof, roof_gather, wm, steps=6):
    """Re-run a few steps with the library's timing mode on (a CUDA event pair around every launch, on the launch stream) and
    restate the two rooflines with the kernels' durations inside the real step — operands where the previous kernel left
    them (the activation matrix is L2-resident there) — instead of the isolated, L2-flushed launch."""
    def one(i):
        flush.zero_()
        train_step(resident[i % len(resident)])
    rows = _profile_rows(cabi, one, steps)
    total = sum(us for _, us in rows.values())
    gemm_us = sum(us for nm, (_, us) in rows.items() if "k_gemm_3xtf32" in nm or "k_sgemm" in nm)
    fam = wm["gemm_flops_per_step"] / (gemm_us / steps * 1e-6) / 1e12 if gemm_us else None
    roof["isolated"] = {"achieved": roof["achieved"], "frac": roof["frac"], "us_per_launch": roof["us_per_launch"], "kernel": roof["kernel"]}
    if fam is not None:
        roof.update(kernel="tcgen05 3xTF32 GEMM family of the step (fwd + dgrad + split-K wgrad of every Linear): total algorithmic "
                           "flops / total in-step kernel time", achieved=fam, frac=fam / roof["peak"], us_per_step=gemm_us / steps,
                    share_of_step=gemm_us / total,
                    timing="sum over %d training steps of every GEMM launch's CUDA-event duration (library timing mode)" % steps,
                    note="fp32-equivalent flops; 3xTF32 spends 3 tf32 MACs per fp32 MAC and dense tf32 is half of bf16, so the ceiling of "
                         "this scheme is peak/6 = %.0f TFLOP/s (achieved/ceiling = %.3f)" % (roof["peak"] / 6, fam / (roof["peak"] / 6)))
        roof.pop("us_per_launch", None)
    gk = wm["gather_kernel"]
    c = [(cnt, us) for nm, (cnt, us) in rows.items() if gk in nm]
    if c:
        cnt, us = sum(a for a, _ in c), sum(b for _, b in c)
        avg = us / cnt
        roof_gather["isolated_us_per_launch"] = roof_gather["us_per_launch"]
        roof_gather["us_per_launch"] = avg
        roof_gather["achieved"] = roof_gather["algorithmic_bytes"] / (avg * 1e-6) / 1e9
        roof_gather["frac"] = roof_gather["achieved"] / roof_gather["peak"]
        roof_gather["timing"] = "average of %d launches inside %d training steps; the activations are L2-resident there" % (cnt, steps)
        roof_gather["share_of_step"] = sum(b for nm, (a, b) in rows.items() if "k_aggregate" in nm or "k_gat_" in nm) / total
    agg = {}
    for nm, (_, us) in rows.items():
        agg[_short(nm)] = agg.get(_short(nm), 0.0) + us
    roof["step_kernels_us"] = {k: round(v / steps, 1) for k, v in sorted(agg.items(), key=lambda kv: -kv[1])[:12]}
    roof["step_sum_us_serialised"] = round(total / steps, 1)  # library kernels only, each bracketed by events (no PDL overlap)


def kernel_rooflines(ops, config, b, dev, wm):
    """Isolated timings (CUDA events on the launch stream, L2 flushed before each launch) of the two kernels the step is made
    of: the config's largest forward GEMM (tensor-bound) and its neighbour gather (HBM/L2-bound)."""
    pk = peaks()
    tr = measured_traffic()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    if config == "contextpred":
        x_key, ei_key, ea_key = "x_substruct", "edge_index_substruct", "edge_attr_substruct"
    else:
        x_key, ei_key, ea_key = "x", "edge_index", "edge_attr"
    n, e = int(b[x_key].shape[0]), int(b[ei_key].shape[1])
    g = ops.Graph(b[ei_key], n)
    M, N, K = wm["top_gemm"]

    def avg_ms(fn, reps=20):
        fn(); torch.cuda.synchronize()
        tot = 0.0
        for _ in range(reps):
            flush.zero_()
            a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); c.record(); c.synchronize()
            tot += a.elapsed_time(c)
        return tot / reps

    with torch.no_grad():
        a = torch.randn(M, K, device=dev)
        w1, b1 = torch.randn(N, K, device=dev) * 0.05, torch.zeros(N, device=dev)
        t_gemm = avg_ms(lambda: ops._linear_fwd(a, w1, b1, True))
        if config == "bio_supervised":
            S = g.summary("bio", ops.AGG_SUM, b[ea_key])
            x, T = torch.randn(n, EMB, device=dev), torch.randn(10, EMB, device=dev)
            t_gather = avg_ms(lambda: ops.aggregate(x, T, g, S, ops.AGG_SUM, concat=True))
        elif config == "gat":
            xl, att = torch.randn(n, 2 * EMB, device=dev), torch.randn(1, 2, 2 * EMB, device=dev) * 0.05
            T, bias = torch.randn(9, 2 * EMB, device=dev) * 0.05, torch.zeros(EMB, device=dev)
            t_gather = avg_ms(lambda: ops.gat(xl, att, T, b[ea_key], g, bias))
        else:
            mode = {"gcn": ops.AGG_GCN, "graphsage": ops.AGG_MEAN}.get(config, ops.AGG_SUM)
            S = g.summary("chem", mode, b[ea_key])
            x, T = torch.randn(n, EMB, device=dev), torch.randn(9, EMB, device=dev)
            t_gather = avg_ms(lambda: ops.aggregate(x, T, g, S, mode))
    gbytes = wm["gather_bytes_per_launch"]
    gflop = 2.0 * M * N * K
    mode = ops.get_precision()
    ach = gflop / (t_gemm * 1e-3) / 1e12
    roof = {"bound": "tensor", "kernel": "largest forward Linear of the step [%d,%d]x[%d,%d] + bias + ReLU (%s)" % (M, K, K, N, mode),
            "achieved": ach, "peak": pk["tensor"], "unit": "TFLOP/s", "frac": ach / pk["tensor"],
            "traffic": tr.get(config, {}).get("gemm", {}).get("dram_bytes_per_launch"),
            "traffic_source": tr.get(config, {}).get("gemm", {}).get("source"),
            "peak_source": pk["src"] + " cuBLAS bf16 dense burst (MEASURED_PEAKS.json)",
            "note": "fp32-equivalent flops; ceiling of the 3xTF32 scheme = peak/6 = %.0f TFLOP/s (achieved/ceiling = %.3f)"
                    % (pk["tensor"] / 6, ach / (pk["tensor"] / 6)),
            "us_per_launch": t_gemm * 1e3}
    roof_g = {"bound": "hbm", "kernel": "%s (gather + segment reduce, one layer pass)" % wm["gather_kernel"],
              "achieved": gbytes / (t_gather * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
              "frac": gbytes / (t_gather * 1e-3) / 1e9 / pk["hbm"],
              "traffic": tr.get(config, {}).get("gather", {}).get("dram_bytes_per_launch"),
              "traffic_source": tr.get(config, {}).get("gather", {}).get("source"),
              "peak_source": pk["src"], "us_per_launch": t_gather * 1e3, "algorithmic_bytes": gbytes}
    return roof, roof_g


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="masking", choices=CONFIG_NAMES)
    ap.add_argument("--precision", default=None, choices=[None, "fp32", "tf32x3"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's loss and gradients to DIR/<name>.npy (B200 arm)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.config == "bio_supervised" else 50
    rank, world, local_rank = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the B200 arm's outputs (--impl b200)")
        run_reference(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
