#!/usr/bin/env python
"""bench.py -- the measurement contract.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c4|c1|c3|c2|mlp|c5]
                    [--dump-outputs DIR]

Default workload (``config.workload``): BASELINE.json configs[3], the C4 sweep at its largest size -- 2^20 independent
pendulum trajectories x 200 save points, Float32 state / Float64 time -- per GPU (weak scaling: every rank integrates its
own slice, no data-path collective).  A "step" is one pass of the hot path over that batch: the forward solve
(``ldeq_solve_fwd``) followed by the pullback of a cotangent (``ldeq_solve_bwd``) in the library's DEFAULT sensitivity
mode, which is the reference's own: ``ForwardDiffSensitivity`` = two dual-number re-solves per trajectory
(pendulum.jl:11).  ``value`` = trajectory-steps/s (B*(T-1) saved grid intervals per solve) with the inputs resident in
HBM; ``e2e`` = the same through ``ldeq_solve_fwd_bwd_host`` from ONE caller thread with pinned host buffers, copies
inside the timed region.  The cheaper discrete adjoint (explicit opt-in) is reported under ``discrete_adjoint``; a C5
data-parallel training step (samples/s, gradient all-reduce measured, fused-vs-NCCL parity self-test) under
``training``; the LatentODE configurations (BASELINE.json configs[1] at batch 256 on the resident exact path -- forward,
forward + discrete adjoint, forward + the reference's InterpolatingAdjoint -- and the tcgen05 path at batch 18 944)
under ``latentode``; ``e2e.link_roofline`` is the host link's ceiling measured in the same run (the step's byte counts as
plain concurrent pinned copies).  ``--impl reference`` times the CPU oracle (the reference is pure Julia, which this image does not have:
the oracle port is the reference arm) on the host cores, same workload, same sizes, same gradient semantics.

One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "latent trajectory-steps/sec (forward solve + gradient, the reference's ForwardDiffSensitivity semantics)"
UNIT = "traj-steps/s"
WORKLOADS = {
    # name: (B per GPU, T, rhs kind, description)
    "c4": (1 << 20, 200, 0, "C4 sweep: 2^20 pendulum trajectories x 200 save points (t = 0:0.05:9.95), forward solve + gradient, "
                            "adaptive Tsit5 abstol 1e-6 reltol 1e-3, fp32 state / fp64 time"),
    "c3": (1024, 50, 1, "C3: pendulum with friction, B = 1024, T = 50, forward solve + gradient"),
    "c1": (64, 50, 0, "C1: friction-less pendulum tutorial shape, B = 64, T = 50, forward solve + gradient"),
}
SENSE_DESC = ("ForwardDiffSensitivity (pendulum.jl:11): 1 primal + 2 dual-number solves per trajectory, partials in the error "
              "norm -- the library default (LDEQ_SENSE_FORWARD_DUAL) and what the reference arm computes")
CPU_BUDGET_S = 150.0   # wall-clock bound of the CPU arm's timed steps
TRAIN_GB, TRAIN_T = 65536, 50   # C5: global batch, frames per sequence
DUMP_TRAJ_SAMPLE = 16384        # --dump-outputs: trajectories of the [T, B, z] result kept (the files stay under 64 MB)


def workload_config(name, B, T):
    """The `config` object: identical on the GPU arm and the reference arm (same workload, same sizes, same gradient)."""
    return {"workload": WORKLOADS[name][3], "trajectories_per_gpu": B, "save_points": T, "gradient": SENSE_DESC,
            "sharding": f"independent trajectories, {B} per GPU, no data-path collective (GOKU.jl:111: prob_func indexes column i)",
            "l2": "inputs larger than L2 (1.68 GB cotangent + 1.68 GB trajectories per step vs 126 MB L2)" if B * T * 8 > (1 << 28)
                  else "working set smaller than L2: an L2-sized buffer is rewritten between timed steps"}


def pendulum_inputs(B, seed=333):
    """create_data.jl:19-22 distribution; PCG64 seed 333 (model_train.jl:42)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    z0 = np.stack([rng.uniform(-np.pi / 6, np.pi / 6, B), rng.uniform(-np.pi / 3, np.pi / 3, B)], 1).astype(np.float32)
    th = rng.uniform(1.0, 2.0, (B, 1)).astype(np.float32)
    return z0, th


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def profile_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/traffic.json)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p)).get(kernel)
    except Exception:
        return None


def issue_roofline(kernels, launch_ms, sm_mhz, sms=148):
    """The instruction-issue roofline of kernels that are bound by it: warp instructions per launch (counted by ncu,
    profiles/traffic.json `issue_model`; the count is a property of the code and the inputs, not of the run) over the
    live launch time, against one warp instruction per SM sub-partition per cycle at the sampled SM clock."""
    model = profile_traffic("issue_model") or {}
    try:
        inst = sum(model[k]["warp_inst"] for k in kernels)
        peak = sms * 4 * float(sm_mhz) * 1e6
        ach = inst / (launch_ms * 1e-3)
        return {"bound": "issue", "achieved": ach / 1e12, "peak": peak / 1e12, "unit": "T warp-inst/s", "frac": ach / peak,
                "warp_inst_per_launch": inst, "lanes_per_inst": [model[k]["lanes"] for k in kernels],
                "source": "instruction counts from profiles/traffic.json (ncu), time and clock measured live"}
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def host_cores() -> int:
    """All the host threads this process may use (torchrun exports OMP_NUM_THREADS=1, which must not throttle the CPU arm)."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_oracle_throughput(B, T, rhs, steps=1, warmup=0, nthreads=0, budget_s=CPU_BUDGET_S):
    """The reference arm / cpu_baseline: the CPU oracle (C++/OpenMP restatement of the reference algorithm:
    per-trajectory Tsit5 under EnsembleThreads, gradients as ForwardDiffSensitivity computes them = 1 primal
    + 2 dual solves per trajectory) timed on the host cores.  Stops early when the wall-clock budget is spent.
    Returns (traj-steps/s, ms per step, cores, steps done)."""
    from oracle import goku as og
    og.build()
    nthreads = nthreads or host_cores()
    z0, th = pendulum_inputs(B)
    t = 0.05 * np.arange(T)
    d = np.random.default_rng(334).standard_normal((T, B, 2)).astype(np.float32)
    for _ in range(warmup):
        og.solve(rhs, z0[:4096], th[:4096], t, nthreads=nthreads)
        og.grad(rhs, z0[:4096], th[:4096], t, d[:, :4096], norm_partials=True, nthreads=nthreads)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        og.solve(rhs, z0, th, t, nthreads=nthreads)
        og.grad(rhs, z0, th, t, d, norm_partials=True, nthreads=nthreads)
        times.append(time.perf_counter() - t0)
        if sum(times) + times[-1] > budget_s:
            break
    dt = float(np.mean(times))
    return B * (T - 1) / dt, dt * 1e3, nthreads, len(times)


def cpu_training_hot_path(Bs=4096, T=TRAIN_T, reps=2):
    """The hot-path part of one C5 training step on the host cores, the way the reference runs it: solve + ForwardDiff
    pullback (oracle, OpenMP), ELBO reduction with its gradient and one ADAMW update (numpy restatements, oracle/loss.py)
    on a bounded sample of `Bs` sequences.  The encoder / decoder layers are NOT included (out of the hot path)."""
    from oracle import goku as og
    from oracle import loss as ol
    z0, th = pendulum_inputs(Bs, seed=1)
    t = 0.05 * np.arange(T)
    rng = np.random.default_rng(0)
    x = rng.random((T, Bs, 784), dtype=np.float32)
    xh = rng.random((T, Bs, 784), dtype=np.float32)
    mus = [rng.standard_normal((Bs, 16)).astype(np.float32) for _ in range(2)]
    lvs = [0.1 * rng.standard_normal((Bs, 16)).astype(np.float32) for _ in range(2)]
    n = 503387
    prm, g = (rng.standard_normal(n).astype(np.float32) for _ in range(2))
    opt = ol.ADAMW(1e-3, (0.9, 0.999), np.float32(0.001))
    d = rng.standard_normal((T, Bs, 2)).astype(np.float32)
    nth = host_cores()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        og.solve(0, z0, th, t, nthreads=nth)
        og.grad(0, z0, th, t, d, norm_partials=True, nthreads=nth)
        ol.loss_batch(x, xh, mus, lvs, 0.5)
        ol.loss_batch_grads(x, xh, mus, lvs, 0.5)
        opt.update("flat", prm, g)
        ts.append(time.perf_counter() - t0)
    dt = min(ts)
    return {"value": Bs / dt, "unit": "samples/s", "ms_per_step": dt * 1e3, "cores": nth, "kind": "port",
            "sample": f"{Bs} of {TRAIN_GB} sequences x {T} frames",
            "scope": "hot-path part of a training step only (latent solve + ForwardDiff pullback + ELBO + its gradient + ADAMW); "
                     "the dense / recurrent encoder-decoder layers are not included, so this is an upper bound for the reference"}


def run_reference(args):
    """`--impl reference`: rank 0 only; the reference's algorithm (CPU oracle, Julia is unavailable) on the host cores, on the
    same workload, sizes and gradient semantics as the GPU arm; the number of timed steps is bounded by a wall-clock budget."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B, T, rhs, desc = WORKLOADS[args.workload]
    val, ms, cores, done = cpu_oracle_throughput(B, T, rhs, steps=max(1, args.steps), warmup=1)
    sample = (f"all {B} trajectories of one GPU's share per step, {done} timed steps of the {args.steps} requested "
              f"(wall-clock budget {CPU_BUDGET_S:.0f} s), {cores} host threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": done,
        "warmup": 1, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, B, T),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "note": "CPU restatement of the reference algorithm (Julia unavailable in this image); "
                                 "optimistic stand-in for Julia+Zygote (no per-trajectory allocation or AD overhead)"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.workload == "c4" and not args.no_training:
        try:
            line["training"] = cpu_training_hot_path()
        except Exception as e:  # noqa: BLE001
            line["training"] = {"unavailable": repr(e)}
    print(json.dumps(line))


def _bind_numa(local):
    """Run this rank (and first-touch its pinned staging buffers) on the NUMA node its GPU hangs off, when the box exposes
    more than one; returns a short description for the record."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = torch.cuda.get_device_properties(local).pci_domain_id
        dev = torch.cuda.get_device_properties(local).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return "numa node unknown"
        cpus = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        want = set()
        for part in cpus.split(","):
            lo, _, hi = part.partition("-")
            want.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        use = want & allowed
        if use and use != allowed:
            os.sched_setaffinity(0, use)
            return f"bound to numa node {node} ({len(use)} cpus)"
        return f"numa node {node} (no rebinding needed)"
    except Exception as e:  # noqa: BLE001
        return f"numa binding skipped: {type(e).__name__}"


def dump_outputs(path, traj, dz0, dtheta, max_traj=DUMP_TRAJ_SAMPLE):
    """`--dump-outputs DIR`: what a caller of the timed path receives from its last step, as .npy files, so that two
    builds can be compared output for output on identical inputs.  traj.npy is the [T, n, z] trajectories
    (ldeq_solve_fwd) of all B trajectories, or, when B > max_traj, of the fixed sample
    sort(default_rng(0).choice(B, max_traj, replace=False)); dz0.npy [B, z] and dtheta.npy [B, p] are the whole gradient
    (ldeq_solve_bwd).  At the C4 size that is 26 + 8 + 4 MB."""
    import torch
    B = traj.shape[1]
    if B > max_traj:
        idx = np.sort(np.random.default_rng(0).choice(B, max_traj, replace=False))
        traj = traj[:, torch.from_numpy(idx).to(traj.device)]
    os.makedirs(path, exist_ok=True)
    for name, a in (("traj", traj), ("dz0", dz0), ("dtheta", dtheta)):
        np.save(os.path.join(path, f"{name}.npy"), a.cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist

    import latentdiffeq_jl_b200 as ldeq

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = _bind_numa(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, T, rhs, desc = WORKLOADS[args.workload]
    K, W = args.steps, max(args.warmup, 3)

    z0n, thn = pendulum_inputs(B, seed=333 + rank)
    t = 0.05 * np.arange(T)
    z0 = torch.from_numpy(z0n).to(dev)
    th = torch.from_numpy(thn).to(dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(334 + rank)
    dtraj = torch.randn(T, B, 2, device=dev, generator=gen)
    h = ldeq.handle(local)
    small = B * T * 8 <= (1 << 28)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if small else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if world > 1:
            tt = torch.tensor([x], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())
        return float(x)

    def device_leg(opts, K, W, sample_clocks=False):
        """K timed steps of (forward solve recording what the pullback needs, pullback); CUDA events around every kernel
        group, the total between two barriers."""
        def step(ev=None):
            if flush is not None:
                flush.fill_(1)
            if ev:
                ev[0].record()
            traj, _, tape = ldeq.goku_solve_raw(z0, th, t, rhs, opts, want_tape=True, want_stats=False)
            tape.p_dim = 1
            if ev:
                ev[1].record()
            g = ldeq.goku_bwd_raw(tape, dtraj)
            if ev:
                ev[2].record()
            tape.free()
            return traj, g
        for _ in range(W):
            step()
        barrier()
        sampler = ClockSampler(local) if (rank == 0 and sample_clocks) else None
        if sampler:
            sampler.start()
        l0 = h.launch_count()
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
        out = None
        barrier()
        for i in range(K):
            out = step(evs[i])
            if i < K - 1:
                out = None   # only the last step's results are kept
        barrier()
        launches = h.launch_count() - l0
        clocks = sampler.stop() if sampler else None
        fwd_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in evs]))
        bwd_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in evs]))
        # the step = the two kernel groups (the L2 flush of a small workload sits outside the event pairs)
        total_ms = allmax(float(np.sum([e[0].elapsed_time(e[2]) for e in evs])))
        rec = {"ms_per_step": total_ms / K, "fwd_ms": fwd_ms, "bwd_ms": bwd_ms, "launches": int(launches), "clocks": clocks}
        return rec, out

    # headline: the library default = the reference's own gradient (dual-number re-solves)
    opts_fd = ldeq.default_opts()
    assert opts_fd.sensealg == ldeq.SENSE_FORWARD_DUAL
    fd, fd_out = device_leg(opts_fd, K, W, sample_clocks=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, fd_out[0], *fd_out[1])
    del fd_out
    value = world * B * (T - 1) / (fd["ms_per_step"] * 1e-3)
    # the explicit opt-in: discrete adjoint of the taped accepted steps
    opts_da = ldeq.default_opts(sensealg=ldeq.SENSE_DISCRETE_ADJOINT)
    da, _ = device_leg(opts_da, K, W)

    # ---- end to end through the host-buffer C-ABI entry points, ONE caller thread, pinned host memory -----------------
    hz0 = torch.from_numpy(z0n).pin_memory()
    hth = torch.from_numpy(thn).pin_memory()
    hd = torch.empty(T, B, 2, dtype=torch.float32).pin_memory()
    hd.copy_(dtraj)
    htraj = torch.empty(T, B, 2, dtype=torch.float32).pin_memory()
    hdz0 = torch.empty(B, 2, dtype=torch.float32).pin_memory()
    hdth = torch.empty(B, 1, dtype=torch.float32).pin_memory()

    def e2e_leg(opts, combined, Ke):
        def one():
            if combined:   # ldeq_solve_fwd_bwd_host: cotangent slabs up while trajectory slabs come down
                ldeq.goku_fwd_bwd_host(hz0, hth, t, hd, rhs, opts, device=local, out=htraj, dz0=hdz0, dtheta=hdth)
            else:          # ldeq_solve_fwd_host, then ldeq_solve_bwd_host (what a training step calls)
                _, tape = ldeq.goku_solve_host(hz0, hth, t, rhs, opts, device=local, want_tape=True, out=htraj)
                ldeq.goku_bwd_host(tape, hd, hdz0, hdth)
                tape.free()
            return float(hdz0[0, 0]) + float(htraj[-1, 0, 0])  # the step's results are read on the host
        for _ in range(2):
            one()
        barrier()
        w0 = time.perf_counter()
        for _ in range(Ke):
            one()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - w0) * 1e3 / Ke
        barrier()
        return allmax(ms)

    def link_probe(reps=4):
        """The ceiling of the end-to-end call at this rank count: the step's own byte counts as plain pinned copies, upload
        and download CONCURRENTLY on two streams, all ranks at once (they share the host's memory system and PCIe root)."""
        up, down = torch.cuda.Stream(), torch.cuda.Stream()
        dbuf_in, dbuf_out = torch.empty_like(dtraj), torch.empty_like(dtraj)
        ms = []
        for i in range(reps + 1):
            torch.cuda.synchronize()
            barrier()
            w0 = time.perf_counter()
            with torch.cuda.stream(up):
                dbuf_in.copy_(hd, non_blocking=True)
            with torch.cuda.stream(down):
                htraj.copy_(dbuf_out, non_blocking=True)
            up.synchronize()
            down.synchronize()
            if i:
                ms.append((time.perf_counter() - w0) * 1e3)
        return allmax(float(np.median(ms)))

    Ke = max(4, min(K, 10))
    link_ms = link_probe()
    e2e_comb = e2e_leg(opts_fd, True, Ke)
    e2e_sep = e2e_leg(opts_fd, False, Ke)
    e2e_da_comb = e2e_leg(opts_da, True, Ke)
    h2d = (hz0.numel() + hth.numel() + hd.numel()) * 4
    d2h = (htraj.numel() + hdz0.numel() + hdth.numel()) * 4

    line = None
    if rank == 0:
        peak, peak_src = measured_peak()
        # algorithmic bytes (SURVEY.md 8(d)): forward reads (z+p) s and writes T z s per trajectory; a pullback reads the
        # cotangent T z s (+ z0, theta) and writes its gradient.  Tape traffic is implementation overhead, not counted.
        alg_fwd = B * (12 + 8 * T)
        alg_bwd = B * (8 * T + 12 + 12)
        alg_fd = 2 * B * (8 * T + 12) + B * 12     # two dual solves, each streams the cotangent once
        fwd_gbs = alg_fwd / (fd["fwd_ms"] * 1e-3) / 1e9
        fdp_gbs = alg_fd / (fd["bwd_ms"] * 1e-3) / 1e9
        bwd_gbs = alg_bwd / (da["bwd_ms"] * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": fd["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, B, T),
            "clocks": fd["clocks"],
            "e2e": {"value": world * B * (T - 1) / (e2e_comb * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_comb, "steps": Ke, "host_threads": 1, "numa": numa,
                    "link_roofline": {"bound": "host link (PCIe + host memory, shared by the ranks of the box)",
                                      "probe": "the step's cotangent upload and trajectory download as plain pinned cudaMemcpyAsync on two "
                                               "streams, concurrently, on all ranks at once (max over ranks, median of 4)",
                                      "probe_ms": link_ms, "peak": world * (h2d + d2h) / (link_ms * 1e-3) / 1e9,
                                      "achieved": world * (h2d + d2h) / (e2e_comb * 1e-3) / 1e9, "unit": "GB/s (both directions, all ranks)",
                                      "frac": link_ms / e2e_comb},
                    "path": "ldeq_solve_fwd_bwd_host (one call, one caller thread, pinned host buffers; batch cut into column slabs, "
                            "cotangent upload / trajectory download / kernels overlapped on the library's own streams)",
                    "separate_calls": {"value": world * B * (T - 1) / (e2e_sep * 1e-3), "ms_per_step": e2e_sep,
                                       "path": "ldeq_solve_fwd_host then ldeq_solve_bwd_host (the pair a training step calls: the "
                                               "cotangent exists only after the forward result is back on the host)"}},
            "gpu_launches": fd["launches"],
            "roofline": {"bound": "hbm", "limiter": "instruction issue",
                         "kernel": "tsit5_fwdsens_kernel (theta-seeded NP=1 + u0-seeded NP=2 launches of one pullback)",
                         "achieved": fdp_gbs, "peak": peak, "unit": "GB/s", "frac": fdp_gbs / peak,
                         "peak_source": peak_src, "launch_ms": fd["bwd_ms"], "algorithmic_bytes_per_launch": alg_fd,
                         "traffic": profile_traffic("tsit5_fwdsens_kernels"),
                         "issue": issue_roofline(("tsit5_fwdsens_kernel_theta", "tsit5_fwdsens_kernel_u0"), fd["bwd_ms"],
                                                 fd["clocks"].get("sm_mhz")),
                         "note": "the dominant kernels of the headline step; the dual solves restate the reference's arithmetic "
                                 "literally (Float64-promoted stage updates, Julia's Float32 sin/cos in Float64): ~1e5 issued "
                                 "instructions per trajectory for 1.6 kB of cotangent -- instruction-issue bound, not HBM bound; "
                                 "see issue_model"},
            "kernels": {
                "tsit5_fwd_kernel<PendulumRHS<float,0>,float,TAPE=1>": {
                    "bound": "hbm", "achieved": fwd_gbs, "peak": peak, "unit": "GB/s", "frac": fwd_gbs / peak, "launch_ms": fd["fwd_ms"],
                    "algorithmic_bytes_per_launch": alg_fwd, "traffic": profile_traffic("tsit5_fwd_kernel_tape"),
                    "issue": issue_roofline(("tsit5_fwd_kernel_tape",), fd["fwd_ms"], fd["clocks"].get("sm_mhz"))},
                "tsit5_bwd_kernel<PendulumRHS<float,0>,float>": {
                    "bound": "hbm", "achieved": bwd_gbs, "peak": peak, "unit": "GB/s", "frac": bwd_gbs / peak, "launch_ms": da["bwd_ms"],
                    "algorithmic_bytes_per_launch": alg_bwd, "traffic": profile_traffic("tsit5_bwd_kernel"),
                    "issue": issue_roofline(("tsit5_bwd_kernel",), da["bwd_ms"], fd["clocks"].get("sm_mhz"))}},
            "issue_model": profile_traffic("issue_model"),
            "discrete_adjoint": {
                "sensealg": "LDEQ_SENSE_DISCRETE_ADJOINT (explicit opt-in: exact derivative of the primal discretisation; equals the "
                            "reference's gradient only within the solver tolerance)",
                "value": world * B * (T - 1) / (da["ms_per_step"] * 1e-3), "unit": UNIT, "ms_per_step": da["ms_per_step"],
                "fwd_ms": da["fwd_ms"], "bwd_ms": da["bwd_ms"], "gpu_launches": da["launches"],
                "e2e": {"value": world * B * (T - 1) / (e2e_da_comb * 1e-3), "ms_per_step": e2e_da_comb}},
        }
        if world == 1 and not args.no_cpu:
            Bs = min(B, 1 << 18)
            val, ms, cores, _ = cpu_oracle_throughput(Bs, T, rhs, steps=1, warmup=1)
            line["cpu_baseline"] = {
                "value": val, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"{Bs} of {B} trajectories (same T={T}), forward + ForwardDiff-style gradient "
                          f"(1 primal + 2 dual solves per trajectory), {ms:.0f} ms"}
    # ---- C5: GOKU-net data-parallel training step around the hot path (samples/s; gradient all-reduce measured) --------
    if args.workload == "c4" and not args.no_training:
        del dtraj, hd, htraj, flush
        torch.cuda.empty_cache()
        tr = training_record(ldeq, dev, world, rank, local, steps=max(3, min(K, 8)), warmup=3)
        if rank == 0:
            line["training"] = tr
            # ---- the LatentODE configurations (BASELINE.json configs[1] and the tcgen05 batch): rank 0, a few seconds ------
            try:
                torch.cuda.empty_cache()
                line["latentode"] = latentode_subrecord(dev)
            except Exception as e:  # the headline record must survive a failure of this appendix
                line["latentode"] = {"unavailable": repr(e)}
        if world > 1:
            dist.barrier()
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def synthetic_frames(theta_angle, device):
    """Synthetic 28x28 pendulum frames [T, B, 784] in [0, 1]: a Gaussian blob at the bob position
    19*(cos(pi/2 + x), sin(pi/2 + x)) px from the pivot (geometry of create_data.jl:27,67-101; Luxor is unavailable)."""
    import torch
    T, B = theta_angle.shape
    ys, xs = torch.meshgrid(torch.arange(28, device=device, dtype=torch.float32),
                            torch.arange(28, device=device, dtype=torch.float32), indexing="ij")
    out = torch.empty(T, B, 784, device=device)
    for lo in range(0, B, 8192):   # in slices: the (T, B, 784) intermediates of one expression would need 4x the output
        a = theta_angle[:, lo:lo + 8192]
        cx = 13.5 + 9.5 * torch.cos(torch.pi / 2 + a)
        cy = 5.0 + 9.5 * torch.sin(torch.pi / 2 + a)
        d2 = (xs.reshape(1, 1, -1) - cx.unsqueeze(-1)) ** 2 + (ys.reshape(1, 1, -1) - cy.unsqueeze(-1)) ** 2
        out[:, lo:lo + 8192] = torch.exp(-d2 / (2 * 1.5 ** 2))
    return out


def training_record(ldeq, dev, world, rank, local, steps, warmup, GB=TRAIN_GB, T=TRAIN_T):
    """BASELINE.json configs[4] / metric M2: GOKU-net data-parallel training, default architecture (GOKU.jl:199-274, 503 387
    parameters), global batch 65 536 pendulum sequences of 50 frames cut into contiguous slices (strong scaling), loss =
    mean over the GLOBAL batch, ONE gradient all-reduce of the flat fp32 bucket per step, identical AdamW on every rank
    (model_train.jl:186-208 run data-parallel).  Both exchange routes are timed: NCCL all-reduce + AdamW kernel, and the
    all-reduce fused with AdamW over NVLink peer memory.  Before timing, the two routes take one step from identical
    weights on identical data and must agree (the multi-rank parity self-test); a mismatch fails the run."""
    import torch
    import torch.distributed as dist

    lo, hi = ldeq.shard_bounds(GB, rank, world)
    Bl = hi - lo
    t = 0.05 * np.arange(T)
    z0n, thn = pendulum_inputs(GB, seed=1)
    with torch.no_grad():   # synthetic data: true pendulum angles from the hot path itself, rasterised on the device
        ang, _, _ = ldeq.goku_solve_raw(torch.from_numpy(z0n[lo:hi]).to(dev), torch.from_numpy(thn[lo:hi]).to(dev), t, 0)
        x = synthetic_frames(ang[..., 0], dev)
    h = ldeq.handle(local)

    def make(symmetric):
        torch.manual_seed(333)   # same initial weights on every rank and for every route
        mt = ldeq.GOKU_basic()
        enc, dec = ldeq.default_layers(mt, 784, ldeq.Pendulum(), device=dev)
        model = ldeq.LatentDiffEqModel(mt, enc, dec)
        flat = ldeq.FlatParams(model, symmetric=symmetric)
        return model, flat, ldeq.ADAMW(flat, 1e-3, (0.9, 0.999), 1e-3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(v):
        if world > 1:
            tt = torch.tensor(v, device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return [float(a) for a in tt]
        return [float(a) for a in v]

    routes = [("nccl", False)] + ([("fused", True)] if world > 1 else [])
    built = {name: make(sym) for name, sym in routes}
    rec = {"metric": "GOKU-net training samples/sec", "unit": "samples/s", "scaling": "strong", "global_batch": GB, "per_gpu_batch": Bl,
           "frames_per_sequence": T, "params": int(built["nccl"][1].n), "gradient": "library default (ForwardDiffSensitivity dual solves)",
           "layers": "encoder / decoder dense layers: stock PyTorch fp32 (outside the hot path); recurrent pattern extractor (forward + "
                     "back-propagation through time), solve, pullback, sample, ELBO, all-reduce + AdamW: libldeq.so"}
    # ---- multi-rank parity self-test: fused peer-memory route vs NCCL route, one step from identical state ----
    if world > 1:
        torch.manual_seed(1234)
        ldeq.train_step(*built["nccl"], x, t, beta=0.5, variational=False, global_batch=GB)
        ldeq.train_step(*built["fused"], x, t, beta=0.5, variational=False, global_batch=GB)
        a, b = built["nccl"][1].flat[:built["nccl"][1].n], built["fused"][1].flat[:built["fused"][1].n]
        err = float((a - b).abs().max() / a.abs().max())
        # replicas must also be identical ACROSS ranks after the step
        chk = torch.stack([a.double().sum(), b.double().sum()])
        lo_, hi_ = chk.clone(), chk.clone()
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
        spread = float((hi_ - lo_).abs().max())
        errs = allmax([err, spread])
        rec["selftest"] = {"fused_vs_nccl_max_rel_param_diff_after_one_step": errs[0], "replica_checksum_spread_across_ranks": errs[1],
                           "ranks": world, "pass": bool(errs[0] <= 1e-5 and errs[1] == 0.0)}
        if not rec["selftest"]["pass"]:
            raise RuntimeError(f"multi-rank parity self-test failed: {rec['selftest']}")
    for name, _ in routes:
        model, flat, opt = built[name]
        tm = {}
        for _ in range(warmup):
            ldeq.train_step(model, flat, opt, x, t, beta=0.5, variational=True, global_batch=GB)
        barrier()
        l0 = h.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        segs = []
        e0.record()
        for _ in range(steps):
            tm = {}
            loss = ldeq.train_step(model, flat, opt, x, t, beta=0.5, variational=True, global_batch=GB, timers=tm)
            segs.append(tm)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) / steps
        def seg(a, b):
            return float(np.mean([s[a].elapsed_time(s[b]) for s in segs]))
        fwd, bwd, xch = seg("start", "loss"), seg("loss", "backward"), seg("backward", "update")
        ms, fwd, bwd, xch = allmax([ms, fwd, bwd, xch])
        rec[name] = {"value": GB / (ms * 1e-3), "ms_per_step": ms, "steps": steps,
                     "forward_ms": fwd, "backward_ms": bwd, "allreduce_adamw_us": xch * 1e3,
                     "libldeq_launches_per_step": (h.launch_count() - l0) / steps, "loss": float(loss),
                     "exchange": ("local AdamW kernel (one GPU: no exchange)" if world == 1 else
                                  "ncclAllReduce of the 2.0 MB flat fp32 bucket + AdamW kernel" if name == "nccl" else
                                  "ONE kernel: all-reduce over NVLink peer memory fused with AdamW (+ 2 symmetric-memory barriers)")}
    best = max((rec[n]["value"], n) for n, _ in routes)
    rec["value"], rec["route"] = best
    del built, x
    torch.cuda.empty_cache()
    return rec


def run_training(args):
    """`--workload c5`: only the training record (see training_record)."""
    import torch
    import torch.distributed as dist

    import latentdiffeq_jl_b200 as ldeq

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rec = training_record(ldeq, dev, world, rank, local, steps=args.steps, warmup=max(args.warmup, 3), GB=args.global_batch)
    if rank == 0:
        print(json.dumps({
            "metric": rec["metric"], "value": rec["value"], "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": rec[rec["route"]]["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "C5: GOKU-net pendulum data-parallel training, default architecture", "global_batch": args.global_batch},
            "gpu_launches": int(rec[rec["route"]]["libldeq_launches_per_step"] * args.steps), "training": rec}))
    if world > 1:
        dist.destroy_process_group()


def _latentode_inputs(workload):
    """Flux-default weights of nODE.jl:14-16 (glorot_uniform, zero bias) packed in Flux.destructure order."""
    B = 256 if workload == "c2" else 18944
    T, dims = 50, [16, 200, 200, 16]
    rng = np.random.Generator(np.random.PCG64(1))
    parts = []
    for i in range(3):
        lim = np.sqrt(6.0 / (dims[i] + dims[i + 1]))
        W = rng.uniform(-lim, lim, (dims[i + 1], dims[i])).astype(np.float32)
        parts += [W.T.reshape(-1), np.zeros(dims[i + 1], np.float32)]
    p = np.concatenate(parts).astype(np.float32)
    z = (0.5 * rng.standard_normal((B, 16))).astype(np.float32)
    d = rng.standard_normal((T, B, 16)).astype(np.float32)
    return B, T, dims, p, z, d, 0.05 * np.arange(T)


def latentode_cpu_oracle(workload, reps=3, max_B=2048):
    """The numpy restatement of the reference's LatentODE path (oracle/mlp.py: BLAS matmuls on the (D,B) state, the way
    Flux Dense layers run on the CPU), forward solve with the batch-global norm + discrete adjoint, on the host cores.
    Bounded sample: at most max_B trajectories of the workload."""
    from oracle import mlp as om

    B, T, dims, p, z, d, t = _latentode_inputs(workload)
    Bs = min(B, max_B)
    z, d = z[:Bs], d[:, :Bs]
    try:  # numpy's BLAS reads OMP_NUM_THREADS (1 under torchrun) at import: give it the host cores
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=host_cores())
    except Exception:
        pass
    om.solve(z, p, dims, t, norm_mode="global")  # warm-up
    t0 = time.perf_counter()
    for _ in range(reps):
        om.solve(z, p, dims, t, norm_mode="global")
    fwd = (time.perf_counter() - t0) / reps
    t0 = time.perf_counter()
    for _ in range(reps):
        _, _, _, tape = om.solve(z, p, dims, t, norm_mode="global", record=True)
        om.discrete_adjoint(p, dims, t, tape, d)
    both = (time.perf_counter() - t0) / reps
    return {"B": Bs, "fwd_ms": fwd * 1e3, "fwd_bwd_ms": both * 1e3, "traj_steps_per_s": Bs * (T - 1) / fwd,
            "traj_steps_per_s_fwd_bwd": Bs * (T - 1) / both, "cores": host_cores()}


def run_latentode_reference(args):
    """`--impl reference --workload c2|mlp`: the CPU oracle of the LatentODE path on the host cores (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    r = latentode_cpu_oracle(args.workload, reps=max(1, min(args.steps, 3)))
    B, T = (256 if args.workload == "c2" else 18944), 50
    line = {"impl": "reference", "metric": "latent trajectory-steps/sec (LatentODE forward solve)", "value": r["traj_steps_per_s"],
            "unit": UNIT, "n_gpus": args.gpus, "steps": max(1, min(args.steps, 3)), "warmup": 1, "ms_per_step": r["fwd_ms"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{'C2' if args.workload == 'c2' else 'MLP sweep'}: LatentODE, MLP RHS 16-200-200-16, batch {B}, T = {T}, "
                                   "adaptive Tsit5 abstol 1e-6 reltol 1e-3, forward solve", "trajectories_per_step": r["B"]},
            "cpu_baseline": {"value": r["traj_steps_per_s"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                             "sample": f"{r['B']} of {B} trajectories per step, numpy/BLAS restatement of the reference algorithm "
                                       "(Julia unavailable in this image)", "fwd_bwd_ms": r["fwd_bwd_ms"]},
            "e2e": {"value": r["traj_steps_per_s"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


LATENTODE_VARIANTS = (("tcgen05_bf16x3_global", dict(norm_mode=0, mlp_math=1)), ("tcgen05_bf16x3_per_traj", dict(norm_mode=1, mlp_math=1)),
                      ("exact_fp32_global", dict(norm_mode=0)), ("exact_fp32_per_traj", dict(norm_mode=1)),
                      # the reference's own reverse pass (NeuralODE default InterpolatingAdjoint): continuous adjoint on
                      # [lambda; mu], ~700 backward steps at C2 against 12 taped forward steps
                      ("exact_fp32_global_interpolating_adjoint", dict(norm_mode=0, sensealg="interpolating_adjoint")))


def latentode_variants(workload, dev, K, W, only=None):
    """Times the LatentODE solve (forward; forward + reverse pass) for the kernel variants of `workload` ('c2' | 'mlp')."""
    import torch

    import latentdiffeq_jl_b200 as ldeq

    B, T, dims, p_np, z_np, d_np, t = _latentode_inputs(workload)
    p, z, d = (torch.from_numpy(a).to(dev) for a in (p_np, z_np, d_np))
    peak_bf16 = 1634.1
    try:
        peak_bf16 = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
    except Exception:
        pass
    h = ldeq.handle(dev.index or 0)
    res = {}
    launches = 0
    for name, kw in LATENTODE_VARIANTS:
        if only is not None and name not in only:
            continue
        kw = dict(kw)
        if kw.get("sensealg") == "interpolating_adjoint":
            kw["sensealg"] = ldeq.SENSE_INTERPOLATING_ADJOINT
        o = ldeq.default_opts(**kw)

        def fwd_bwd():
            tr, st, tape = ldeq.mlp_solve_raw(z, p, dims, t, o, want_tape=True)
            g = ldeq.mlp_bwd_raw(tape, d)
            tape.free()
            return st
        try:
            for _ in range(W):
                tr, st, _ = ldeq.mlp_solve_raw(z, p, dims, t, o)
                fwd_bwd()
        except ldeq.LdeqError as e:
            res[name] = {"unavailable": str(e)}
            continue
        torch.cuda.synchronize()
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        l0 = h.launch_count()
        e0.record()
        for _ in range(K):
            tr, st, _ = ldeq.mlp_solve_raw(z, p, dims, t, o)
        e1.record()
        for _ in range(K):
            fwd_bwd()
        e2.record()
        torch.cuda.synchronize()
        launches += h.launch_count() - l0
        ms, ms2 = e0.elapsed_time(e1) / K, e1.elapsed_time(e2) / K
        att = float((st.naccept + st.nreject).float().mean())
        rhs = B * (6 * att + 2)
        res[name] = {"ms": ms, "fwd_bwd_ms": ms2, "traj_steps_per_s": B * (T - 1) / (ms * 1e-3),
                     "traj_steps_per_s_fwd_bwd": B * (T - 1) / (ms2 * 1e-3), "rk_steps_per_traj_per_s": B * att / (ms * 1e-3),
                     "naccept_mean": float(st.naccept.float().mean()), "algorithmic_tflops": rhs * 92800 / (ms * 1e-3) / 1e12}
        if "tcgen05" in name:
            # tensor-pipe work actually issued: padded widths (208) and three bf16 passes per product
            issued = rhs * 3 * 2 * (16 * 208 + 208 * 208 + 208 * 16) / (ms * 1e-3) / 1e12
            res[name]["roofline"] = {"bound": "tensor", "achieved": issued, "peak": peak_bf16, "unit": "TFLOP/s",
                                     "frac": issued / peak_bf16, "traffic": None,
                                     "note": "bf16 flops issued to tcgen05 (3 passes, padded widths) / measured cuBLAS bf16 peak"}
            # reverse pass (ldeq_mlp_tc_bwd.cu): per accepted step and stage one recomputed evaluation, one transposed
            # (input-gradient) evaluation and one weight-gradient contraction of the same shape, each in 3 bf16 passes
            na = float(st.naccept.float().mean())
            issued_b = B * na * 7 * 3 * 3 * 2 * (16 * 208 + 208 * 208 + 208 * 16) / (max(ms2 - ms, 1e-6) * 1e-3) / 1e12
            res[name]["roofline_reverse_pass"] = {"bound": "tensor", "achieved": issued_b, "peak": peak_bf16, "unit": "TFLOP/s",
                                                  "frac": issued_b / peak_bf16, "ms": ms2 - ms, "traffic": None,
                                                  "note": "adjoint kernel (recompute + transposed products) + split-K weight-gradient "
                                                          "GEMM + reduce, all tcgen05; bf16 flops issued / measured cuBLAS bf16 peak"}
    return B, T, res, launches


def latentode_subrecord(dev):
    """The LatentODE configurations in the default bench line (rank 0): C2 (BASELINE.json configs[1], B = 256) on the exact
    resident path -- forward, forward + discrete adjoint, forward + the reference's InterpolatingAdjoint -- and the same
    network at B = 18 944 on tcgen05 (forward, forward + tcgen05 reverse pass)."""
    out = {"metric": "LatentODE solve, MLP right-hand side 16-200-200-16, T = 50, adaptive Tsit5 (abstol 1e-6, reltol 1e-3), batch-global norm"}
    _, _, c2, _ = latentode_variants("c2", dev, 5, 3, only=("exact_fp32_global", "exact_fp32_global_interpolating_adjoint"))
    ex, ia = c2.get("exact_fp32_global", {}), c2.get("exact_fp32_global_interpolating_adjoint", {})
    out["c2_batch_256"] = {"forward_ms": ex.get("ms"), "forward_discrete_adjoint_ms": ex.get("fwd_bwd_ms"),
                           "forward_interpolating_adjoint_ms": ia.get("fwd_bwd_ms", ia.get("unavailable")),
                           "traj_steps_per_s": ex.get("traj_steps_per_s")}
    _, _, big, _ = latentode_variants("mlp", dev, 5, 3, only=("tcgen05_bf16x3_global",))
    tc = big.get("tcgen05_bf16x3_global", {})
    out["batch_18944_tcgen05"] = {"forward_ms": tc.get("ms"), "forward_reverse_pass_ms": tc.get("fwd_bwd_ms", tc.get("unavailable")),
                                  "traj_steps_per_s": tc.get("traj_steps_per_s"), "roofline": tc.get("roofline"),
                                  "roofline_reverse_pass": tc.get("roofline_reverse_pass")}
    return out


def run_latentode(args):
    """`--workload c2` (BASELINE.json configs[1]: LatentODE, small-MLP RHS 16-200-200-16, batch 256, T = 50) and
    `--workload mlp` (the same network at batch 18 944 = 128 trajectories per SM: where batch x hidden is a genuine
    dense contraction).  Adaptive Tsit5, per-trajectory and global (reference) error norm, exact CUDA-core path vs the
    tcgen05 path; forward solve and forward + adjoint.  Unit: trajectory-steps/s (and accepted RK steps per trajectory
    per second, SURVEY.md 8(d) C2)."""
    import torch

    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    K, W = args.steps, max(args.warmup, 3)
    B, T, res, launches = latentode_variants(args.workload, dev, K, W)
    best = max((v["traj_steps_per_s"], k) for k, v in res.items() if "ms" in v)
    line = {"metric": "latent trajectory-steps/sec (LatentODE forward solve)", "value": best[0], "unit": UNIT, "n_gpus": 1,
            "steps": K, "warmup": W, "ms_per_step": res[best[1]]["ms"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{'C2' if args.workload == 'c2' else 'MLP sweep'}: LatentODE, MLP RHS 16-200-200-16, batch {B}, T = 50, "
                                   "adaptive Tsit5 abstol 1e-6 reltol 1e-3, forward solve", "best": best[1]},
            "gpu_launches": launches, "variants": res}
    tc = [v["roofline"] for k, v in res.items() if "roofline" in v]
    if tc:
        line["roofline"] = max(tc, key=lambda r: r["frac"])
    if not args.no_cpu:
        r = latentode_cpu_oracle(args.workload)
        line["cpu_baseline"] = {"value": r["traj_steps_per_s"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                "sample": f"{r['B']} of {B} trajectories, numpy/BLAS restatement of the reference algorithm, forward solve "
                                          "with the batch-global norm", "fwd_ms": r["fwd_ms"], "fwd_bwd_ms": r["fwd_bwd_ms"]}
    print(json.dumps(line))


def main():
    # the contract is ONE JSON line on stdout: libraries that print there (NCCL's version banner, warnings) are sent to
    # stderr for the whole run, and the JSON line goes to the real stdout
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    _orig_print = print

    def emit(*a, **k):
        sys.stdout.flush()
        os.write(real_stdout, (" ".join(str(x) for x in a) + "\n").encode())
    globals()["print"] = emit
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS) + ["c5", "c2", "mlp"])
    ap.add_argument("--global-batch", type=int, default=65536, help="c5 only")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-training", action="store_true", help="skip the C5 training sub-record of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the trajectories and gradients of the last timed step as DIR/*.npy "
                                                          "(GOKU workloads c1, c3, c4; rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload not in WORKLOADS):
        ap.error(f"--dump-outputs needs --impl ours and a workload of {sorted(WORKLOADS)}")
    if args.workload in ("c2", "mlp"):
        if args.impl == "reference":
            run_latentode_reference(args)
        else:
            run_latentode(args)
    elif args.workload == "c5":
        if args.impl == "reference":
            if int(os.environ.get("RANK", "0")) == 0:
                r = cpu_training_hot_path()
                print(json.dumps({"impl": "reference", "metric": "GOKU-net training samples/sec", "value": r["value"], "unit": "samples/s",
                                  "n_gpus": args.gpus, "steps": 2, "warmup": 0, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                                  "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                                  "config": {"workload": "C5: GOKU-net pendulum data-parallel training, default architecture",
                                             "global_batch": args.global_batch},
                                  "cpu_baseline": r, "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0,
                                                             "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        else:
            run_training(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
