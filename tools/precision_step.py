"""Training-step throughput of the four precision modes on the bench workload, and per-launch convolution times of the
three tensor-core modes.

    python tools/precision_step.py [--steps 20] [--warmup 5] [--rounds 2] [--out profiles/r03_precision_modes.json]

Workload: bench.py's default (dune3d encoder + heads, 64 events per step, Trainer, a pool of 4 distinct batches resident
on the device).  Modes are alternated ("fp32", "mixed", "tf32", "bf16", then again), each round on a fresh Trainer:
warm-up steps, then bench.settle_allocator until a chunk of steps allocates no device memory, then `steps` timed steps
between two CUDA events.  For "mixed", "tf32" and "bf16" one more profiled step (ops.set_profiler: CUDA events around
every C-ABI call) gives the per-launch forward / dgrad / wgrad times of every convolution shape of the step (median over
the layers of a shape): the 3^3 submanifold layers, the 2^3 downsamples, the stem and the bottleneck of the six levels.
The card name and power limit are read in the same process.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

MODES = ("fp32", "mixed", "tf32", "bf16")
PROFILED = ("mixed", "tf32", "bf16")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def level_times(recs):
    """{kind: {"K x n_in x n_out": median us}} of the convolution launches of one profiled step."""
    out = {}
    for r in recs:
        if not r["kind"].startswith("conv_"):
            continue
        key = f"{r['K']} x {r['n_in']} x {r['n_out']} ({r['rows_out']} rows)"
        out.setdefault(r["kind"], {}).setdefault(key, []).append(r["ms"] * 1000.0)
    return {k: {s: round(float(np.median(v)), 1) for s, v in d.items()} for k, d in out.items()}


def run_mode(mode, pool, args, dev):
    import sparseconvnet as scn
    from bench import settle_allocator
    from sparseeventid_b200.scn import ops
    from sparseeventid_b200.trainer import Trainer
    scn.set_precision(mode)
    trainer = Trainer(scn, "dune3d", device=dev, seed=0)
    tuples = [b for b, _ in pool]

    def step(i):
        return trainer.step(tuples[i % len(pool)], pool[i % len(pool)][1], prefetch=tuples[(i + 1) % len(pool)])

    for i in range(args.warmup):
        step(i)
    settled = settle_allocator(step, lambda: int(torch.cuda.memory_stats(dev).get("num_device_alloc", 0)),
                               lambda flag: flag, chunk=4)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        loss = step(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    res = {"mode": mode, "ms_per_step": round(ms, 3), "events_per_s": round(args.batch * 1000.0 / ms, 1),
           "settle_steps": settled, "loss": float(loss.detach())}
    if mode in PROFILED:
        prof = ops.Profiler()
        ops.set_profiler(prof)
        if hasattr(torch.cuda, "_sleep"):
            torch.cuda._sleep(60_000_000)            # the host runs ahead: event pairs time kernels, not launches
        step(0)
        ops.set_profiler(None)
        res["conv_us"] = level_times(prof.finish())
    del trainer
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_precision_modes.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "precision_step.py needs a CUDA device"
    from bench import host_batch
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    pool = []
    for i in range(4):
        c, f, bs, lab = host_batch(args.batch, 1234 + 1000 * i, "dune3d")
        pool.append(((torch.from_numpy(c).to(dev), torch.from_numpy(f).to(dev), bs),
                     {k: torch.from_numpy(v).to(dev) for k, v in lab.items()}))
    runs = []
    for r in range(args.rounds):
        for mode in MODES:
            res = run_mode(mode, pool, args, dev)
            res["round"] = r
            runs.append(res)
            print(json.dumps({k: v for k, v in res.items() if k != "conv_us"}), flush=True)
    summary = {m: {"events_per_s": [x["events_per_s"] for x in runs if x["mode"] == m],
                   "ms_per_step": [x["ms_per_step"] for x in runs if x["mode"] == m]} for m in MODES}
    out = {"card": card(), "workload": f"dune3d default encoder + heads, {args.batch} events per step, Trainer, pool of 4 "
           f"resident batches; {args.warmup} warm-up steps + allocator settled, {args.steps} timed steps per mode per "
           f"round, modes alternated over {args.rounds} rounds; CUDA events",
           "summary": summary, "runs": runs}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps({"card": out["card"], "summary": summary}))


if __name__ == "__main__":
    main()
