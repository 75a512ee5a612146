"""Eager ``train_step`` against ``GraphedTrainStep`` on one GPU.

    python scripts/bench_graph_step.py [--batches 64,8192] [--steps 500] [--block 25] [--warmup 20] [--out DIR]

Workloads: the default GOKU-net (``default_layers``, Pendulum, adaptive Tsit5, ForwardDiffSensitivity, fused logits ELBO,
AdamW) on 784-pixel ``bench.synthetic_frames`` of T = 50 frames, at the reference's batch of 64 (BASELINE.md C1) and at
8192 as a no-regression check.  Both modes train the same model in one process, alternating blocks of ``--block`` steps
until each has run ``--steps``; every block is timed with CUDA events (the step time of a block is its time over its
steps).  Writes ``graph_step.json`` under ``--out`` with the median and spread of the step time and samples/s per mode, the
libldeq kernel launches of one eager step, and the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import latentdiffeq_jl_b200 as ldeq  # noqa: E402
from bench import pendulum_inputs, synthetic_frames  # noqa: E402

T = 50
P_IN = 784


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clk = ([s.strip() for s in q.stdout.strip().split(",")] + ["", "", ""])[:3] if q.returncode == 0 else ("", "", "")
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi_name": name, "power_limit_w": power, "max_sm_clock_mhz": clk}


def stats(ms_per_step, batch):
    a = np.asarray(ms_per_step)
    sps = batch / (a * 1e-3)
    return {"step_ms_median": float(np.median(a)), "step_ms_p10": float(np.percentile(a, 10)), "step_ms_p90": float(np.percentile(a, 90)),
            "step_ms_min": float(a.min()), "step_ms_max": float(a.max()), "samples_per_s_median": float(np.median(sps)),
            "samples_per_s_p10": float(np.percentile(sps, 10)), "samples_per_s_p90": float(np.percentile(sps, 90)), "blocks": len(a)}


def run(batch, steps, block, warmup, dev):
    torch.manual_seed(333)
    z0, th = pendulum_inputs(batch + 64, seed=1)
    with torch.no_grad():
        ang, _, _ = ldeq.goku_solve_raw(torch.from_numpy(z0).to(dev), torch.from_numpy(th).to(dev), 0.05 * np.arange(T + 16), ldeq.RHS_PENDULUM)
        frames = synthetic_frames(ang[..., 0], dev)            # [T + 16, batch + 64, 784]
    t = 0.05 * np.arange(T)
    rng = np.random.default_rng(0)

    def batch_at(k):   # a different window of frames each step, without host work inside the timed loop
        o, b = int(rng.integers(0, 16)), int(rng.integers(0, 64))
        return frames[o:o + T, b:b + batch]

    xs = [batch_at(k).contiguous() for k in range(8)]
    enc, dec = ldeq.default_layers(ldeq.GOKU_basic(), P_IN, ldeq.Pendulum(), device=dev)
    model = ldeq.LatentDiffEqModel(ldeq.GOKU_basic(), enc, dec)
    flat = ldeq.FlatParams(model)
    opt = ldeq.ADAMW(flat, 1e-3, (0.9, 0.999), 1e-3)
    graphed = ldeq.GraphedTrainStep(model, flat, opt, xs[0], t)
    eager = lambda x, beta: ldeq.train_step(model, flat, opt, x, t, beta)
    h = ldeq.handle(0)
    n0 = h.launch_count()
    eager(xs[0], 0.5)
    torch.cuda.synchronize()
    launches = h.launch_count() - n0
    for k in range(warmup):
        eager(xs[k % 8], 0.5)
        graphed(xs[k % 8], 0.5)
    torch.cuda.synchronize()
    times = {"eager": [], "graph": []}
    done = 0
    while done < steps:
        for mode, fn in (("eager", eager), ("graph", graphed)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(block):
                loss = fn(xs[k % 8], 0.5)
            e1.record()
            e1.synchronize()
            times[mode].append(e0.elapsed_time(e1) / block)
        done += block
    assert torch.isfinite(loss).all()
    out = {"batch": batch, "T": T, "pixels": P_IN, "steps_per_mode": done, "block": block,
           "eager": stats(times["eager"], batch), "graph": stats(times["graph"], batch), "libldeq_launches_per_eager_step": launches}
    out["speedup_median"] = out["eager"]["step_ms_median"] / out["graph"]["step_ms_median"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="64,8192")
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--block", type=int, default=25)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default="graph_step_bench")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_graph_step.py measures on a CUDA device; there is none")
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "workloads": [run(int(b), args.steps, args.block, args.warmup, dev) for b in args.batches.split(",")]}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "graph_step.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "workloads": [{k: w[k] for k in ("batch", "speedup_median")} | {
        "eager_ms": w["eager"]["step_ms_median"], "graph_ms": w["graph"]["step_ms_median"]} for w in res["workloads"]]}))


if __name__ == "__main__":
    main()
