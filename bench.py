#!/usr/bin/env python
"""bench.py -- 3D sparse ResNet (recipes/dune3d.yaml encoder + heads) TRAINING events/s on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one full training step of the hot path over one batch of synthetic DUNE-shaped events:
InputLayer (hash + row numbering) -> rulebooks -> 56 sparse convolutions + 53 BatchNorms ... ->
SparseToDense -> heads -> focal loss -> backward -> gradient all-reduce (N>1) -> Adam.
Workload at N=1 = BASELINE.json configs[2] per GPU ("3D sparse ResNet training, event-sharded data
parallel, batch 64/GPU, bf16 tensor-core convs"); weak scaling (64 events on every rank).

Prints ONE JSON line (rank 0).  `value` = events/s with the batch already resident in HBM;
`e2e` = events/s through the public module API starting from pinned HOST buffers: every step copies one batch
(SCN input tuple + labels) host -> device on a copy stream, one step ahead like a data loader, and copies its loss
device -> host into pinned memory (consumed one step later).  Both loops tell the trainer which batch comes next so
that its rulebooks are built during the current backward (--no-prefetch disables that).  `roofline` describes the dominant kernel family (the
gather-GEMM convolution kernels), timed live with CUDA events on the launching stream in a separate
instrumented pass after the timed region.  `cpu_baseline` = the oracle port of SparseConvNet's CPU
algorithm on the host cores, on a bounded sample.  `--impl reference` times that CPU arm alone.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch
import torch.distributed as dist

METRIC = "3D sparse ResNet train events/sec"
METRIC_2D = "2D multiplane sparse ResNet train events/sec"   # --dataset dune2d (BASELINE.json configs[1])
UNIT = "events/s"
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            d["_source"] = "measured"
            return d
        except Exception:
            pass
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback"
    return d


# ------------------------------------------------------------------------------------------- data


def host_batch(batch, seed, dataset, raw=False):
    """Synthetic larcv batch -> SCN input tuple exactly as the reference's transform produces it
    (coords float64 [N,4] with the batch index last, features float32 [N,1]) + 4 label vectors
    (+ the raw -999-padded larcv batch-filler array itself with raw=True)."""
    from sparseeventid_b200 import synthetic
    from sparseeventid_b200.data_transforms import larcvsparse_to_scnsparse_2d, larcvsparse_to_scnsparse_3d
    arr = synthetic.larcv_batch_3d(batch, seed=seed) if dataset == "dune3d" else synthetic.larcv_batch_2d(batch, seed=seed)
    coords, feats, bs = larcvsparse_to_scnsparse_3d(arr) if dataset == "dune3d" else larcvsparse_to_scnsparse_2d(arr)
    labels = synthetic.make_labels(batch, seed=seed)
    out = (np.ascontiguousarray(coords, dtype=np.float64), np.ascontiguousarray(feats, dtype=np.float32), bs, labels)
    return out + (arr,) if raw else out


# ns of step time per active site of resolution level l (B200, measured per-level kernel times of the bench step
# divided by the level's rows: convolutions fwd + dgrad + wgrad and BatchNorm; the two deepest levels are latency-bound
# and do not depend on their row counts)
LEVEL_COST_NS = (6.1, 11.0, 22.6, 35.0)


def event_cost(arr, dataset):
    """Cost proxy of every event of a larcv batch array [n][planes][voxels][D+1]: the sum over the resolution levels of
    (active sites of the level) x (measured ns per site).  Equal level-0 voxel counts still leave the step times of the
    ranks +-6% apart (8 GPUs: the slowest rank cost 1.3 ms of a 20 ms step) because the deeper levels' sizes depend on
    how the event is spread in space; their site counts follow from the coordinates alone (floor(x / 2^l), unique)."""
    from sparseeventid_b200 import synthetic
    n = arr.shape[0]
    cost = np.zeros(n)
    for e in range(n):
        for pl in range(arr.shape[1]):
            v = arr[e, pl]
            live = v[:, -1] != synthetic.PAD
            c = v[live, :-1].astype(np.int64)
            if c.shape[0] == 0:
                continue
            if dataset == "dune2d":                  # 2-D planes: [1,2,2] downsampling, the plane axis is not strided
                c = c[:, -2:]
            for l, w in enumerate(LEVEL_COST_NS):
                q = c >> l
                key = q[:, 0]
                for a in range(1, q.shape[1]):
                    key = key * 65536 + q[:, a]
                cost[e] += w * np.unique(key).shape[0]
    return cost


def balanced_host_batch(batch, world, rank, seed, dataset, raw=False):
    """Event-sharded data parallelism with work balancing (SURVEY.md 8e): the global batch of batch x world events
    is dealt to the ranks in a snake over the events sorted by a cost proxy (event_cost), so every rank gets the same
    number of events AND nearly the same work.  Contiguous sharding of DUNE-like events leaves the heaviest of 8
    ranks 12% above the mean, and a synchronous step runs at the pace of the heaviest rank.  Deterministic: every rank
    generates the same global batch from the seed and keeps its share."""
    from sparseeventid_b200 import synthetic
    from sparseeventid_b200.data_transforms import larcvsparse_to_scnsparse_2d, larcvsparse_to_scnsparse_3d
    n = batch * world
    arr = synthetic.larcv_batch_3d(n, seed=seed) if dataset == "dune3d" else synthetic.larcv_batch_2d(n, seed=seed)
    counts = event_cost(arr, dataset)
    order = np.argsort(-counts, kind="stable")
    mine = []
    for j, e in enumerate(order):
        r = j % (2 * world)
        r = r if r < world else 2 * world - 1 - r
        if r == rank:
            mine.append(int(e))
    mine = np.sort(np.asarray(mine))
    sub = np.ascontiguousarray(arr[mine])
    coords, feats, bs = larcvsparse_to_scnsparse_3d(sub) if dataset == "dune3d" else larcvsparse_to_scnsparse_2d(sub)
    labels = {k: v[mine] for k, v in synthetic.make_labels(n, seed=seed).items()}
    out = (np.ascontiguousarray(coords, dtype=np.float64), np.ascontiguousarray(feats, dtype=np.float32), bs, labels)
    return out + (sub,) if raw else out


class ClockSampler:
    """SM clocks / power / throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line), every
    300 ms.  In-process through NVML (nvidia_ml_py) when it is importable: an `nvidia-smi -lms 100` child process was
    measured to cost the timed loop up to 20% in some runs (2533-2648 vs 3260-3310 events/s in the same build, the e2e
    loop without a sampler stable at 3214-3371); nvidia-smi remains the fallback.  The NVML queries are the same ones
    nvidia-smi makes (clocks.sm, clocks.max.sm, power.draw, clocks_event_reasons)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []
        self.samples = []          # NVML path: (sm MHz, max MHz, watts, reasons bitmask)
        self.nvml = None
        self.stop_flag = False

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.gpu_index])
            except (ValueError, IndexError):
                pass
        return self.gpu_index

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            # the maximum SM clock is a constant of the board: queried ONCE, before the timed region -- under load
            # nvmlDeviceGetMaxClockInfo takes 2 ms (median) to 90 ms and stalls kernel launches meanwhile (it made one
            # step of the timed loop 70-120 ms long in 3 runs of 5); current clock, power and event reasons take ~10 us
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self._physical_index())], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                mode = os.environ.get("SCN_BENCH_SAMPLER", "all")          # diagnostic: which NVML query perturbs the loop
                clk = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM) if mode != "none" else 0
                pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0 if mode in ("all", "power") else 0.0
                rs = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)) if mode in ("all", "reasons") else 0
                self.samples.append((clk, self.max_mhz, pw, rs))
            except Exception:
                pass
            time.sleep(0.3)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=1)
            n = self.nvml
            if not self.samples:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
            bits = {"hw_slowdown": n.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": n.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksEventReasonSwPowerCap}
            reasons = sorted(k for k, b in bits.items() if any(s[3] & b for s in self.samples))
            return {"sm_mhz": float(np.median([s[0] for s in self.samples])), "sm_max_mhz": float(max(s[1] for s in self.samples)),
                    "power_w_max": float(max(s[2] for s in self.samples)), "samples": len(self.samples), "reasons": reasons,
                    "source": "NVML in-process (clock, power, event reasons), every 300 ms; max clock read once before"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(power)),
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------------ CPU arm


def cpu_events_per_s(dataset, events, steps, warmup, seed=1234):
    """Oracle port of SparseConvNet's CPU path (per-offset index_select -> mm -> index_add_) running the
    same encoder + heads + focal loss + Adam, all host threads.  Returns (events/s, seconds/step, cores)."""
    from oracle import sparseconvnet_oracle as oscn
    from sparseeventid_b200 import networks
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    oscn.set_numerics("fp32")
    enc, head = networks.build_networks(oscn, dataset)
    model = networks.EventIDModel(enc, head)
    model.train()
    opt = torch.optim.Adam(model.parameters(), lr=1.0 * 3e-3, eps=1e-6, betas=(0.8, 0.9), weight_decay=1e-6)
    times = []
    for it in range(warmup + steps):
        coords, feats, bs, labels = host_batch(events, seed + 1000 * it, dataset)
        lab = {k: torch.as_tensor(v) for k, v in labels.items()}
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        loss = networks.focal_loss(lab, model((torch.as_tensor(coords), torch.as_tensor(feats), bs)))
        loss.backward()
        opt.step()
        float(loss.detach())
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    sec = float(np.mean(times))
    return events / sec, sec, cores


def workload_config(dataset, batch, n_params, n_voxels, world, sharding, pool):
    """The `config` of BOTH arms (ours and --impl reference): the workload, not how an arm runs it (that is `dtype`,
    `cpu_baseline.sample`, ...)."""
    return {"workload": f"{dataset} default encoder (56 sparse convs) + 4 heads, {n_params / 1e6:.2f}M params, "
                        f"training step, batch {batch} events/GPU",
            "events_per_gpu": batch, "mean_voxels_per_batch": n_voxels, "parallelism": f"dp{world}",
            "sharding": sharding,
            "l2_policy": f"inputs_larger_than_L2 (activations of one step >> 126 MB; {pool} distinct batches cycled)"}


def sharding_text(args, world):
    if world == 1:
        return "one rank"
    if args.same_batches:
        return "identical batches on every rank (diagnostic)"
    if args.no_balance:
        return "contiguous by event"
    return ("by event, dealt in a snake over the order of a per-event cost proxy (sites of resolution levels 0-3 x measured "
            "ns per site): equal events and ~equal work per rank")


def run_reference(args, rank):
    """The CPU arm: the oracle port of SparseConvNet's CPU algorithm (SCN itself is absent from the image: kind
    "port") on the host cores, on OUR arm's config; each step is a bounded sample of that workload (--cpu-events events
    of the batch) so that the run ends within minutes."""
    if rank != 0:
        return
    from oracle import sparseconvnet_oracle as oscn
    from sparseeventid_b200 import networks
    events = args.cpu_events
    world = args.gpus
    enc, head = networks.build_networks(oscn, args.dataset)
    n_params = sum(p.numel() for p in enc.parameters()) + sum(p.numel() for p in head.parameters())
    del enc, head
    n_voxels = int(np.mean([host_batch(args.batch, 1234 + 1000 * i, args.dataset)[0].shape[0] for i in range(args.pool)]))
    v, sec, cores = cpu_events_per_s(args.dataset, events, args.steps, min(args.warmup, 1))
    sample = (f"{events} of the {args.batch} synthetic {args.dataset} events of a batch per step (bounded sample), "
              f"{args.steps} timed steps after {min(args.warmup, 1)} warm-up, fp32, the same training step "
              f"(encoder + heads + focal loss + Adam) through the oracle port of SparseConvNet's CPU algorithm")
    line = {
        "impl": "reference", "metric": METRIC if args.dataset == "dune3d" else METRIC_2D, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": min(args.warmup, 1), "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.dataset, args.batch, n_params, n_voxels, world, sharding_text(args, world), args.pool),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ GPU arm


def conv_algorithmic(rec, elem_bytes):
    """FLOPs / compulsory bytes of one conv launch (SURVEY.md 8d)."""
    P, K, n_in, n_out = rec["pairs"], rec["K"], rec["n_in"], rec["n_out"]
    flops = 2.0 * P * n_in * n_out
    rows_in, rows_out = rec["rows_in"], rec["rows_out"]
    if rec["kind"] == "conv_wgrad":
        by = rows_in * n_in * elem_bytes + rows_out * n_out * elem_bytes + K * n_in * n_out * 4 + 8 * P
    else:
        by = rows_in * n_in * elem_bytes + rows_out * n_out * elem_bytes + K * n_in * n_out * 2 + 8 * P
    return flops, by


def settle_allocator(step, alloc_count, any_rank, chunk, cap=60):
    """Run `step(i)` in chunks of `chunk` steps until a whole chunk passes without a device allocation on ANY rank (or
    `cap` steps).  `any_rank(flag)` is the collective OR of the ranks' flags: every step contains the gradient all-reduce,
    so all ranks must leave this loop after the same number of steps -- a rank-local decision deadlocks the job (N > 1).
    The ranks agree once per chunk, not per step, so that inside a chunk the host runs ahead of the GPU exactly as in the
    timed loops (that is what makes the allocator grow its cache).  Returns the number of steps run."""
    n = 0
    while n < cap:
        before = alloc_count()
        for _ in range(chunk):
            step(n)
            n += 1
        if not any_rank(alloc_count() != before):
            break
    return n


def training_state_reset(trainer, seed=0):
    """Snapshot of the state `trainer` is in now (call it on a freshly constructed one).  Returns a function that puts
    the trainer back into it, in place with a few multi-tensor launches (no allocation; the CUDA-graphed heads keep their
    parameter addresses): the parameters and buffers, zero Adam moments and step counts, the learning-rate schedule at
    step 0, and the random generators reseeded (head dropout).  A step from there computes the same thing in every run,
    however many steps came before."""
    live = list(trainer.model.parameters()) + list(trainer.model.buffers())
    init = [t.detach().clone() for t in live]

    def reset():
        with torch.no_grad():
            torch._foreach_copy_(live, init)
            torch._foreach_zero_([v for st in trainer.opt.state.values() for v in st.values() if torch.is_tensor(v)])
        trainer.sched.last_epoch = -1
        trainer.sched.step()
        trainer.global_step = 0
        torch.manual_seed(seed)
    return reset


DUMP_SAMPLE = 1 << 21          # draws of the seeded sample of parameter / gradient elements that --dump-outputs writes


def step_outputs(trainer, loss):
    """What one training step hands its caller, as float32 host arrays: the loss, the step's gradients and the updated
    parameters, and the BatchNorm running statistics.  Gradients and parameters (all of them concatenated in
    named_parameters order, ~21M elements) are sampled at fixed, seeded positions, the same in every run."""
    def host(tensors):                   # gathered on the host: no device allocation between the timed loops
        return torch.cat([t.detach().reshape(-1).float().cpu() for t in tensors]).numpy()
    params = list(trainer.model.parameters())
    flat_p, flat_g = host(params), host([p.grad for p in params])
    idx = np.unique(np.random.default_rng(0).integers(0, flat_p.size, DUMP_SAMPLE))
    return {"loss": host([loss]), "grad_sample": flat_g[idx], "param_sample": flat_p[idx],
            "bn_running_stats": host([b for b in trainer.model.buffers() if b.is_floating_point()])}


def kernel_source_hash():
    """sha256 of the dominant kernel's sources: ties a committed ncu summary to the build it was captured on."""
    import hashlib
    h = hashlib.sha256()
    for f in ("conv_tc.cu", "tc_ptx.cuh", "common.cuh"):
        with open(os.path.join(ROOT, "sparseeventid_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def run_ours(args, rank, world, local_rank):
    import sparseconvnet as scn
    from sparseeventid_b200 import _lib
    from sparseeventid_b200.scn import ops
    from sparseeventid_b200.trainer import Trainer

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback for the product path)"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    scn.set_precision(args.precision)
    peaks = load_peaks()
    trainer = Trainer(scn, args.dataset, device=dev, seed=0)
    reset_training_state = training_state_reset(trainer) if args.dump_outputs else None
    n_params = sum(p.numel() for p in trainer.model.parameters())
    lib = _lib.lib()

    # ---- inputs: a pool of distinct host batches per rank (pinned), mirrored on the device
    pool = []
    for i in range(args.pool):
        if world > 1 and args.same_batches:          # diagnostic: every rank steps through the SAME batches (no straggler term)
            coords, feats, bs, labels, arr = host_batch(args.batch, 1234 + 1000 * i, args.dataset, raw=True)
        elif world > 1 and not args.no_balance:
            coords, feats, bs, labels, arr = balanced_host_batch(args.batch, world, rank, 1234 + 1000 * i, args.dataset, raw=True)
        else:
            coords, feats, bs, labels, arr = host_batch(args.batch, 1234 + 100000 * rank + 1000 * i, args.dataset, raw=True)
        h = {"coords": torch.from_numpy(coords).pin_memory(), "feats": torch.from_numpy(feats).pin_memory(),
             "labels": {k: torch.from_numpy(v).pin_memory() for k, v in labels.items()}, "bs": bs,
             "larcv": torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()}
        pool.append(h)
    dpool = [{"coords": h["coords"].to(dev), "feats": h["feats"].to(dev),
              "labels": {k: v.to(dev) for k, v in h["labels"].items()}, "bs": h["bs"]} for h in pool]
    n_voxels = int(np.mean([h["coords"].shape[0] for h in pool]))
    # e2e input: the raw larcv batch-filler array (what src/io/larcv_fetcher.py:394-419 hands to the transform), copied as
    # it is and compacted on the GPU (scn_larcv_count / scn_larcv_compact); --e2e-tuple uploads the host-transformed
    # SCN tuple instead (coords float64 [N,4] + features)
    if args.e2e_tuple:
        h2d_bytes = int(np.mean([h["coords"].numel() * 8 + h["feats"].numel() * 4 + 4 * 8 * args.batch for h in pool]))
    else:
        h2d_bytes = int(np.mean([h["larcv"].numel() * 4 + 4 * 8 * args.batch for h in pool]))

    # Both loops tell the trainer which batch comes next (what a data loader with one batch of look-ahead knows), so the
    # next step's rulebooks -- a function of coordinates only -- are built on the rulebook stream during this step's
    # backward (--no-prefetch turns that off).
    tuples = [(d["coords"], d["feats"], d["bs"]) for d in dpool]
    last_loss = [None]

    def step_resident(i):
        d = dpool[i % len(dpool)]
        nxt = None if args.no_prefetch else tuples[(i + 1) % len(dpool)]
        last_loss[0] = trainer.step(tuples[i % len(dpool)], d["labels"], prefetch=nxt).detach()
        return last_loss[0]

    copy_stream = torch.cuda.Stream(device=dev)
    staged = {}
    from sparseeventid_b200.data_transforms import larcvsparse_to_scnsparse_2d_gpu, larcvsparse_to_scnsparse_3d_gpu
    to_scn_gpu = larcvsparse_to_scnsparse_3d_gpu if args.dataset == "dune3d" else larcvsparse_to_scnsparse_2d_gpu

    def upload(i):
        """H2D of step i's inputs from pinned host memory on a copy stream -> (batch tuple, labels, done event)."""
        h = pool[i % len(pool)]
        with torch.cuda.stream(copy_stream):
            if args.e2e_tuple:
                c = h["coords"].to(dev, non_blocking=True)
                f = h["feats"].to(dev, non_blocking=True)
            else:                   # device-side twin of the reference's transform; one row count comes back to the host
                raw_dev = h["larcv"].to(dev, non_blocking=True)
                c, f = to_scn_gpu(raw_dev)[:2]
            lab = {k: v.to(dev, non_blocking=True) for k, v in h["labels"].items()}
            ev = copy_stream.record_event()
        return (c, f, h["bs"]), lab, ev

    def step_e2e(i):
        # this step's inputs: uploaded during the previous step (or now, for the first one); the next step's upload is
        # issued before this step runs so it overlaps it -- every step still copies exactly one batch host -> device
        batch, lab, ev = staged.pop(i) if i in staged else upload(i)
        main = torch.cuda.current_stream(dev)
        main.wait_event(ev)
        for t in [batch[0], batch[1]] + list(lab.values()):
            t.record_stream(main)
        nxt, nxt_ev = None, None
        if not args.no_prefetch and i + 1 < e2e_steps[0]:
            staged[i + 1] = upload(i + 1)
            nxt, nxt_ev = staged[i + 1][0], staged[i + 1][2]
        loss = trainer.step(batch, lab, prefetch=nxt, prefetch_ready=nxt_ev)
        # D2H of the step's result: every step's loss is copied to pinned host memory inside the timed region; the
        # host consumes it one step later (asynchronous logging), so the read-back does not drain the GPU queue
        slot = loss_host[i % 2]
        slot.copy_(loss.detach().reshape(1), non_blocking=True)
        ev_done = main.record_event()
        if loss_pending:
            pev, pslot = loss_pending.pop()
            pev.synchronize()
            losses.append(float(pslot[0]))
        loss_pending.append((ev_done, slot))
        return None

    e2e_steps = [args.steps]
    loss_host = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_pending, losses = [], []

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        import gc
        gc.collect()
        gc.disable()          # the step is close to host/GPU balance: a collection inside the 0.3 s region is visible
        try:
            return _timed(fn, steps)
        finally:
            gc.enable()

    step_times = []
    untimed = []                  # (start, end) events around work inside a timed loop that is not part of a step

    def _timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]      # per-step marks: diagnostics only
        l0 = lib.scn_launch_count()
        e0.record()
        for i in range(steps):
            fn(i)
            marks[i].record()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) - sum(a.elapsed_time(b) for a, b in untimed)
        untimed.clear()
        prev, per_step = e0, []
        for m in marks:
            per_step.append(prev.elapsed_time(m))
            prev = m
        step_times.append([round(v, 2) for v in per_step])
        launches = lib.scn_launch_count() - l0
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, int(launches)

    def note(msg):                                        # progress marks on stderr (stdout carries the one JSON line)
        if world > 1:
            print(f"[bench rank {rank}] {msg}", file=sys.stderr, flush=True)

    note("pool ready, first steps (graph capture of the heads happens here)")
    # setup, not warm-up: every batch of the pool goes through both loops once so that the caching allocator has seen
    # all tensor sizes (a first-time cudaMalloc is a device synchronisation) before the W warm-up steps start
    for i in range(2 * len(dpool)):
        step_resident(i)
    for i in range(len(pool)):
        step_e2e(i)
    staged.clear(); loss_pending.clear(); losses.clear()
    torch.cuda.synchronize()
    # Allocator settling (setup, untimed): rulebook tensors are allocated on the rulebook stream and consumed on the main
    # stream, so the caching allocator may reuse their blocks only after the consuming kernels have finished; with the host
    # a step ahead it cudaMalloc()s new blocks instead -- a device synchronisation, up to several 100 ms for the 248 MB stem
    # table -- until its cache holds enough of them.  Steps are run until a whole cycle of the pool passes without a
    # device allocation on any rank (or 60 steps), so that the timed loops measure the steady state.
    def device_alloc_count():
        return int(torch.cuda.memory_stats(dev).get("num_device_alloc", 0))

    def any_rank(flag):                                   # the ranks must agree on the number of steps: each one all-reduces
        if world == 1:
            return flag
        t = torch.tensor([1.0 if flag else 0.0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return bool(t.item() > 0)

    settle_steps = 0
    for loop in (step_e2e, step_resident):                # the resident loop last: it is the one timed first
        settle_steps += settle_allocator(loop, device_alloc_count, any_rank, chunk=3 * len(dpool))
        torch.cuda.synchronize()
    staged.clear(); loss_pending.clear(); losses.clear()
    note(f"allocator settled after {settle_steps} steps")
    # the clock sampler (nvidia-smi -lms 100) is started BEFORE the warm-up steps: its start-up (process launch, NVML
    # initialisation) takes driver locks for a few hundred ms and was measured to cost the first timed loop up to 15%
    # when it fell inside it (2825 vs 3272 events/s in one process); it keeps sampling through the timed region
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)
    for i in range(args.warmup):
        step_resident(i)
    def device_allocs():
        st = torch.cuda.memory_stats(dev)
        return int(st.get("num_device_alloc", 0)), int(st.get("num_device_free", 0)), int(st.get("num_alloc_retries", 0))
    def step_timed(i):
        # --dump-outputs: the last timed step starts from the trainer's initial state, so that its results depend on the
        # arguments alone (the steps before it carry the last bits of order-dependent sums, which Adam amplifies); the
        # reset is bracketed by events and its interval is left out of the loop's time
        if reset_training_state is not None and i == args.steps - 1:
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record()
            reset_training_state()
            r1.record()
            untimed.append((r0, r1))
        return step_resident(i)
    a0 = device_allocs()
    ms, launches = timed(step_timed, args.steps)
    a1 = device_allocs()
    clocks = sampler.stop() if rank == 0 else None
    # the last timed step's results, taken before the e2e loop trains on
    outputs = step_outputs(trainer, last_loss[0]) if rank == 0 and args.dump_outputs else None
    note(f"resident loop timed: {ms / args.steps:.2f} ms/step")
    ms_e2e, _ = timed(step_e2e, args.steps)
    a2 = device_allocs()
    note(f"e2e loop timed: {ms_e2e / args.steps:.2f} ms/step")
    # cudaMalloc / cudaFree calls of the caching allocator inside the two timed loops (each one is a device synchronisation:
    # a source of isolated slow steps): [resident loop, e2e loop] x [mallocs, frees, retries]
    alloc_events = [[a1[i] - a0[i] for i in range(3)], [a2[i] - a1[i] for i in range(3)]]
    while loss_pending:                                   # the last step's loss (its copy finished inside the timed region)
        pev, pslot = loss_pending.pop()
        pev.synchronize()
        losses.append(float(pslot[0]))
    assert len(losses) == args.steps, "e2e: a loss was not read back"

    value = args.batch * world * args.steps / (ms * 1e-3)
    e2e = args.batch * world * args.steps / (ms_e2e * 1e-3)

    # host time to ENQUEUE one step (stepping thread, GPU queue empty at the start so nothing throttles the host; the
    # rulebooks of the step were prefetched by the step before, as in the timed loops): the step is host-bound when
    # this approaches ms_per_step
    import time as _time
    step_resident(args.steps)                             # seeds the prefetch chain for the measured steps
    host_ms = []
    for i in range(3):
        tr_thread = getattr(trainer, "_join_prefetch", None)
        if tr_thread is not None:
            tr_thread()
        torch.cuda.synchronize()
        t0 = _time.perf_counter()
        step_resident(args.steps + 1 + i)
        host_ms.append((_time.perf_counter() - t0) * 1e3)
    torch.cuda.synchronize()
    host_enqueue_ms = float(np.median(host_ms))

    # ---- instrumented pass (rank 0): CUDA events around every launch of this library's hot kernels
    # (every rank runs the two extra steps -- they contain the gradient all-reduce -- only rank 0 records)
    roof, breakdown = None, None
    prof = ops.Profiler() if rank == 0 else None
    ops.set_profiler(prof)
    for i in range(2):
        # A GPU-side delay first, so that the host (slower here: Python functions + two events per call) is ahead of the
        # GPU for the whole step and the interval between a call's two events is kernel time, not launch latency.
        if hasattr(torch.cuda, "_sleep"):
            torch.cuda._sleep(60_000_000)          # ~30 ms at 1.97 GHz
        step_resident(i)
    ops.set_profiler(None)
    barrier()
    if rank == 0:
        recs = prof.finish()
        eb = 2 if args.precision == "bf16" else 4
        agg = {}
        for r in recs:
            a = agg.setdefault(r["kind"], {"ms": 0.0, "launches": 0, "flops": 0.0, "bytes": 0.0})
            a["ms"] += r["ms"]; a["launches"] += 1
            if r["kind"].startswith("conv"):
                fl, by = conv_algorithmic(r, eb)
                a["flops"] += fl; a["bytes"] += by
            else:
                a["bytes"] += r.get("bytes", 0.0)
        tc = [r for r in recs if r["kind"] in ("conv_fwd", "conv_dgrad") and r["tc"]]
        if tc:
            fl = sum(conv_algorithmic(r, eb)[0] for r in tc)
            by = sum(conv_algorithmic(r, eb)[1] for r in tc)
            t = sum(r["ms"] for r in tc) * 1e-3
            peak = peaks["bf16_tflops_sustained"]
            traffic, traffic_note = None, None
            prof_path = os.path.join(ROOT, "profiles", "r02_conv_tc_ncu_summary.json")
            if os.path.exists(prof_path):      # dram bytes of ONE ncu --set full capture of this kernel (committed)
                pj = json.load(open(prof_path))
                if pj.get("kernel_source_sha256") == kernel_source_hash():
                    traffic = pj.get("traffic_bytes_per_launch")
                    traffic_note = (f"dram read+write of the captured launch ({pj.get('shape')}; its algorithmic bytes: "
                                    f"{pj.get('algorithmic_bytes_per_launch')}); `achieved` averages all conv launches of a step")
                else:                          # a capture of another build says nothing about this run
                    traffic_note = "stale: csrc/conv_tc.cu changed since profiles/r02_conv_tc_ncu_summary.json was captured"
            roof = {"bound": "tensor", "kernel": "gather-GEMM conv fwd/dgrad (k_conv_tc, tcgen05)", "achieved": fl / t / 1e12,
                    "peak": peak, "unit": "TFLOP/s", "frac": fl / t / 1e12 / peak, "traffic": traffic,
                    "traffic_note": traffic_note,
                    "launches": len(tc), "avg_launch_us": t / len(tc) * 1e6,
                    "flops_per_launch": fl / len(tc), "algorithmic_bytes_per_launch": by / len(tc),
                    "achieved_algorithmic_gbs": by / t / 1e9, "hbm_peak_gbs": peaks["hbm_gbs"],
                    "frac_of_hbm": by / t / 1e9 / peaks["hbm_gbs"], "peak_source": peaks["_source"],
                    "share_of_step": sum(r["ms"] for r in tc) / 2 / (ms / args.steps)}
            # per layer shape (the 8 convolutions of a level share it): achieved TFLOP/s, its fraction of the tensor
            # peak and of the launch's binding roof = max(flops / tensor peak, algorithmic bytes / HBM peak)
            per = {}
            for r in tc:
                key = f"{r['kind']} K={r['K']} {r['n_in']}->{r['n_out']} rows={r['rows_out']}"
                a = per.setdefault(key, {"launches": 0, "us": 0.0, "flops": 0.0, "bytes": 0.0})
                fl_r, by_r = conv_algorithmic(r, eb)
                a["launches"] += 1; a["us"] += r["ms"] * 1e3; a["flops"] += fl_r; a["bytes"] += by_r
            roof["per_layer_shape"] = {
                k: {"launches_per_step": v["launches"] / 2, "avg_us": round(v["us"] / v["launches"], 1),
                    "tflops": round(v["flops"] / v["us"] / 1e6, 1), "frac_of_tensor_peak": round(v["flops"] / v["us"] / 1e6 / peak, 4),
                    "frac_of_binding_roof": round(max(v["flops"] / (peak * 1e12), v["bytes"] / (peaks["hbm_gbs"] * 1e9)) / (v["us"] * 1e-6), 4)}
                for k, v in sorted(per.items(), key=lambda kv: -kv[1]["us"])}
            try:
                # per launch the binding roof is max(flops / tensor peak, algorithmic bytes / HBM peak): at these widths
                # (arithmetic intensity below the 207 FLOP/B ridge) it is usually the HBM one (SURVEY.md 8d)
                t_roof = sum(max(conv_algorithmic(r, eb)[0] / (peak * 1e12), conv_algorithmic(r, eb)[1] / (peaks["hbm_gbs"] * 1e9))
                             for r in tc)
                roof["time_at_binding_roof_ms_per_step"] = t_roof * 1e3 / 2
                roof["frac_of_binding_roof"] = t_roof / t
            except Exception:                       # never let a derived figure cost the bench line
                pass
        breakdown = {k: {"ms_per_step": v["ms"] / 2, "launches_per_step": v["launches"] / 2,
                         "tflops": (v["flops"] / (v["ms"] * 1e-3) / 1e12) if v["flops"] and v["ms"] else None,
                         "algorithmic_gbs": (v["bytes"] / (v["ms"] * 1e-3) / 1e9) if v["bytes"] and v["ms"] else None}
                     for k, v in sorted(agg.items(), key=lambda kv: -kv[1]["ms"])}
        if args.breakdown_json:
            with open(args.breakdown_json, "w") as f:
                json.dump({"ms_per_step": ms / args.steps, "breakdown": breakdown,
                           "per_launch": [{k: v for k, v in r.items()} for r in recs[: len(recs) // 2]]}, f, indent=1)

    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, sec, cores = cpu_events_per_s(args.dataset, args.cpu_events, 2, 1)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{args.cpu_events} events/step x 2 timed steps (+1 warm-up) of the same encoder+heads "
                         f"training step through the oracle port of SparseConvNet's CPU algorithm, fp32"}

    if rank == 0:
        line = {
            "metric": METRIC if args.dataset == "dune3d" else METRIC_2D, "value": value, "unit": UNIT, "n_gpus": world,
            "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16" if args.precision != "fp32" else "f32", "data": "synthetic",
            "config": workload_config(args.dataset, args.batch, n_params, n_voxels, world, sharding_text(args, world), args.pool),
            "precision_mode": args.precision,
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": 4,
                    "input": ("host-transformed SCN tuple (coords float64 [N,4], features fp32)" if args.e2e_tuple else
                              "raw larcv batch-filler array [B, planes, 50000, D+1] fp32 (-999 padded) from pinned host memory, "
                              "transformed on the GPU (scn_larcv_count / scn_larcv_compact)"),
                    "d2h": "every step's loss -> pinned host memory inside the timed region, consumed one step later",
                    "loss_first_last": [losses[0], losses[-1]] if losses else None,
                    "losses_finite": bool(np.all(np.isfinite(losses)))},
            "gpu_launches": launches,
            "host_enqueue_ms_per_step": round(host_enqueue_ms, 3),
            "device_mallocs_frees_retries_in_timed_loops": alloc_events,
            "allocator_settle_steps": settle_steps,
            "step_ms_median_max": [[round(float(np.median(t)), 2), round(float(np.max(t)), 2)] for t in step_times],
            "step_ms_resident": step_times[0] if step_times else None,
            "rulebook_ms": round(sum(v["ms_per_step"] for k, v in (breakdown or {}).items() if k.startswith("rulebook")), 3),
            "rulebook_ms_note": "hash build + InputLayer rules + all submanifold / strided neighbour tables of one batch, GPU time on the rulebook stream (overlaps the feature kernels)",
            "roofline": roof,
            "cpu_baseline": cpu,
            "breakdown_ms_per_step": {k: round(v["ms_per_step"], 3) for k, v in (breakdown or {}).items()},
        }
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dataset", default="dune3d", choices=["dune3d", "dune2d"])
    ap.add_argument("--batch", type=int, default=64, help="events per GPU")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "mixed", "fp32"])
    ap.add_argument("--pool", type=int, default=4, help="distinct synthetic batches cycled per rank")
    ap.add_argument("--cpu-events", type=int, default=8, help="events per step of the bounded CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-prefetch", action="store_true", help="do not build the next batch's rulebooks ahead")
    ap.add_argument("--no-balance", action="store_true", help="N>1: contiguous event sharding instead of voxel-count balancing")
    ap.add_argument("--same-batches", action="store_true", help="N>1 diagnostic: identical batches on every rank")
    ap.add_argument("--e2e-tuple", action="store_true", help="e2e uploads the host-transformed SCN tuple instead of the raw larcv array")
    ap.add_argument("--dump-outputs", metavar="DIR", help="start the last timed step from the initial training state and "
                    "write its results (loss, sampled gradients and updated parameters, BatchNorm running statistics) as "
                    "DIR/<name>.npy, float32")
    ap.add_argument("--breakdown-json", metavar="PATH", help="write the per-kernel breakdown of the instrumented pass to PATH")
    args = ap.parse_args()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # 5-minute collective timeout (default 10): a mismatched collective ends the run with an error instead of eating
        # the caller's time budget; the longest legitimate gap between two collectives is the pool generation (tens of s)
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=300))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
