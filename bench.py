#!/usr/bin/env python
"""bench.py - BASELINE.json metric: QP solves/s, batch 4096 Lite3 trot problems (N=10) per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (condense + factor + ADMM, cold start) over one batch
of 4096 synthetic problems per GPU (SURVEY.md section 8d, config 2).  One process per GPU
(torchrun sets RANK/LOCAL_RANK/WORLD_SIZE); problems shard by batch index with no
collective on the solve path ("weak" scaling: 4096 problems per GPU).  Rank 0 prints one
JSON line; its `configs` block carries the other BASELINE configs (3: 65536 mixed-gait problems
sharded over the ranks, 4: N=30 x 16384 per GPU, 5: closed-loop rollouts) and `sharding_check`
the bit-identity of a batch solved sharded over the ranks (NCCL gather) against one GPU.
`--impl reference` times the reference's CPU algorithm (OSQP restatement in C, oracle/) on the
host cores on the FULL 4096-problem batch of the same workload.
`--dump-outputs DIR` writes what the last timed step returned on rank 0 (U, X, iters, pri_res, dua_res,
status; the reference arm: U, iters, status) as DIR/<name>.npy, float32 or float64, with the batch
indices they belong to in problem_index.npy.  The inputs are seeded, so two builds run with the same
arguments can be compared output for output.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# One hardware queue per stream: with the default 8 connections the copy streams of the pipelined host path can
# share a queue, and an event wait at its head (a result copy waiting for its solve) then also holds back the next
# step's input copies: the steps serialise (0.31 instead of 0.23 ms).  Must be set before CUDA is initialised.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

import numpy as np  # noqa: E402

BATCH = 4096
HORIZON = 10
WORKLOAD = "config2: batch 4096 Lite3 trot MPC QPs per GPU, N=10, randomized CoM states/velocity refs, cold start"
KERNEL_SRC = os.path.join(ROOT, "mpc-for-dynamic-locomotion-in-the-mit-cheetah-3_b200", "csrc", "cmpc_kernels.cuh")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--horizon", type=int, default=HORIZON)
    ap.add_argument("--gaits", default="trot")
    ap.add_argument("--cpu-sample", type=int, default=0, help="problems per CPU step (0 = the full batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs 3/4/5 block")
    ap.add_argument("--rollout-ticks", type=int, default=1000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy")
    return ap.parse_args()


DUMP_BYTES = 60 * 10 ** 6      # payload cap of --dump-outputs: 64 MB in all with the index and the .npy headers


def dump_outputs(path, **arrays):
    """Per-problem outputs (leading dim = batch) as path/<name>.npy: floats as they are (float32 / float64),
    integers as float64 (exact).  A batch too large for DUMP_BYTES is cut to a fixed, seeded sample of
    problems; problem_index.npy lists the batch indices written."""
    arrays = {k: np.asarray(v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in arrays.items() if v is not None}
    arrays = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in arrays.items()}
    B = next(iter(arrays.values())).shape[0]
    per_problem = sum(v.nbytes for v in arrays.values()) // B + 8
    idx = np.arange(B)
    if per_problem * B > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(B, DUMP_BYTES // per_problem, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "problem_index.npy"), idx.astype(np.float64))
    for k, v in arrays.items():
        np.save(os.path.join(path, f"{k}.npy"), np.ascontiguousarray(v[idx]))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_source_sha():
    try:
        return hashlib.sha256(open(KERNEL_SRC, "rb").read()).hexdigest()[:16]
    except OSError:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.thr.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                  "sw_power_cap"), r[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def algorithmic_work(N, stance_counts, iters):
    """SURVEY.md section 8(d) work model per solve (averaged over the batch):
    FLOPs = R_f (n^3/3 + 2 n^2) + 12 n^2 + K (2.08 n^2 + 33 n), smem bytes = K 4 n^2,
    HBM bytes = 4 (62 N + 44) + N."""
    n = 3.0 * stance_counts.astype(np.float64)
    K = iters.astype(np.float64)
    flops = (n ** 3 / 3 + 2 * n ** 2) + 12 * n ** 2 + K * (2.08 * n ** 2 + 33 * n)
    smem = K * 4 * n ** 2
    hbm = 4.0 * (62 * N + 44) + N
    return float(flops.mean()), float(smem.mean()), float(hbm)


# ------------------------------------------------------------------------------------------
def run_reference(args):
    """Reference arm: the reference's CPU algorithm (fp64 OSQP restatement, oracle/) on all host
    threads; each step solves the FULL batch of the workload (same config as our arm)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_baseline
    import mpc_b200 as pkg
    sample = args.cpu_sample or args.batch
    pb = pkg.problems.synthetic_batch(args.batch, N=args.horizon, gaits=tuple(args.gaits.split(",")), seed=0)
    pb = pb.slice(0, sample)
    for _ in range(max(min(args.warmup, 2), 1)):
        cpu_baseline.solve_batch(pb.slice(0, min(256, sample)))
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        info = cpu_baseline.solve_batch(pb)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, U=info["U"], iters=info["iters"], status=info["status"])
    tot = sum(times)
    val = sample * args.steps / tot
    what = "the full batch" if sample == args.batch else f"{sample} of the {args.batch} problems"
    line = {
        "impl": "reference", "metric": "QP solves/sec", "value": val, "unit": "solves/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_step": sample, "horizon": args.horizon,
                   "solved_frac": float((info["status"] == 1).mean())},
        "cpu_baseline": {"value": val, "unit": "solves/s", "cores": info["threads"],
                         "kind": info["kind"], "sample": f"{what} per step, all {info['threads']} host threads, "
                         f"mean {info['mean_iters']:.1f} OSQP iterations"},
        "e2e": {"value": val, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


class Bench:
    """Timing helpers of one rank."""

    def __init__(self, torch, dist, dev, world):
        self.torch, self.dist, self.dev, self.world = torch, dist, dev, world
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
        self.stream = torch.cuda.current_stream(dev)

    def barrier(self):
        self.torch.cuda.synchronize(self.dev)
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def timed_steps(self, fn, steps, warmup=3, pre=None):
        """Per-step CUDA-event times (ms) of fn(); L2 flushed (256 MiB fill) before every step."""
        torch = self.torch
        for _ in range(warmup):
            if pre:
                pre()
            fn()
        self.barrier()
        evs = []
        for _ in range(steps):
            if pre:
                pre()
            self.flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(self.stream)
            fn()
            e1.record(self.stream)
            evs.append((e0, e1))
        self.barrier()
        return [a.elapsed_time(b) for a, b in evs]

    def max_over_ranks(self, vals):
        t = self.torch.tensor(vals, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def gather(self, vals):
        """[world][len(vals)] on every rank."""
        t = self.torch.tensor(vals, dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return [[float(v) for v in t]]
        out = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [[float(v) for v in o] for o in out]


def kernel_times(pkg, bench, N, B, local, dargs, out, steps, **opts):
    """Duration of the solve kernel alone: CUDA events recorded by the library on the launching
    stream immediately around that one kernel (cfg.time_kernel), L2 flushed between steps."""
    mpc_t = pkg.BatchedMPC(N=N, max_batch=B, device=local, warm_mode=0, time_kernel=1, **opts)
    ms = []
    for i in range(steps + 3):
        bench.flush.fill_(1)
        mpc_t.solve(*dargs, out=out)
        if i >= 3:
            ms.append(mpc_t.last_kernel_ms)
    bench.barrier()
    mpc_t.close()
    return ms


def per_rank_block(bench, kern_ms, step_ms, iters):
    rows = bench.gather([statistics.mean(kern_ms), statistics.mean(step_ms), float(iters.max()), float(iters.mean())])
    k = [r[0] for r in rows]
    return {"kernel_ms": {"min": min(k), "median": statistics.median(k), "max": max(k), "per_rank": k},
            "step_ms_per_rank": [r[1] for r in rows], "max_iters_per_rank": [int(r[2]) for r in rows],
            "mean_iters_per_rank": [r[3] for r in rows]}


def fp32_frac(flops, B, kern_s, fp32_peak):
    return flops * B / kern_s / fp32_peak


def run_config(pkg, bench, torch, local, rank, world, name, pb, steps, fp32_peak, scaling, global_batch=None):
    """Cold-start solves/s of one more BASELINE config on this rank's problems `pb`."""
    dev = bench.dev
    B, N = pb.B, pb.N
    dargs = [torch.from_numpy(a).to(dev) for a in pb.f32()]
    mpc = pkg.BatchedMPC(N=N, max_batch=B, device=local, warm_mode=0)
    out = mpc.alloc_outputs(B, want_X=True, device=dev)
    step_ms = bench.timed_steps(lambda: mpc.solve(*dargs, out=out), steps)
    iters = out[2].cpu().numpy()
    status = out[5].cpu().numpy()
    mpc.close()
    kern_ms = kernel_times(pkg, bench, N, B, local, dargs, out, steps)
    tmax, = bench.max_over_ranks([sum(step_ms)])
    ranks = per_rank_block(bench, kern_ms, step_ms, iters)
    flops, smem_b, hbm_b = algorithmic_work(N, pb.stance.sum((1, 2)), iters)
    total = (global_batch if global_batch is not None else B * world) * steps
    return {"workload": name, "value": total / (tmax * 1e-3), "unit": "solves/s", "scaling": scaling,
            "batch_this_rank": B, "horizon": N, "ms_per_step": tmax / steps,
            "kernel_ms": statistics.mean(kern_ms),
            "fp32_frac": fp32_frac(flops, B, statistics.mean(kern_ms) * 1e-3, fp32_peak),
            "algorithmic_flop_per_solve": flops, "mean_iters": float(iters.mean()), "max_iters": int(iters.max()),
            "solved_frac": float((status == 1).mean()), "per_rank": ranks}


def sharding_check(pkg, bench, torch, dist, local, rank, world):
    """SURVEY.md section 8e: ONE global batch solved as `world` contiguous shards (one per GPU), the
    results gathered over NCCL with sharding.gather_results, must equal bit for bit what one GPU
    returns for the whole batch (rank 0 solves it alone as the comparison)."""
    Bg, N = 8192, 10
    pb = pkg.problems.synthetic_batch(Bg, N=N, gaits=pkg.problems.GAIT_NAMES, seed=123, mu=(0.3, 1.0))
    mpc = pkg.BatchedMPC(N=N, max_batch=Bg, device=local, warm_mode=0)
    lo, hi, U, X, st = pkg.sharding.solve_sharded(mpc, pb, rank, world, device=bench.dev)
    u0 = U[:, 0, :].contiguous()
    if world > 1:
        g_u0, g_it, g_st = pkg.sharding.gather_results(u0, st.iters, st.status, Bg)
    else:
        g_u0, g_it, g_st = u0, st.iters, st.status
    res = None
    if rank == 0:
        full = [torch.from_numpy(a).to(bench.dev) for a in pb.f32()]
        Uf, _, sf = mpc.solve(*full)
        torch.cuda.synchronize(bench.dev)
        res = {"global_batch": Bg, "shards": world,
               "gather": "sharding.gather_results over NCCL all_gather" if world > 1 else "single rank (no gather)",
               "bit_identical_u0": bool(torch.equal(g_u0, Uf[:, 0, :])),
               "identical_iters": bool(torch.equal(g_it, sf.iters)),
               "identical_status": bool(torch.equal(g_st, sf.status))}
    bench.barrier()
    mpc.close()
    return res


def run_rollout(pkg, bench, torch, local, world, ticks):
    """config 5: closed-loop warm-started rollouts, 8192 robots per GPU, friction sweep 0.3-1.0."""
    B = 8192
    ro = pkg.ClosedLoopRollout(B, N=10, gaits=("trot",), mu=(0.3, 1.0), seed=0, device=local)
    ro.capture(10)
    bench.barrier()
    l0 = ro.mpc.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    done0 = int(ro.tick.item())
    e0.record(bench.stream)
    ro.run(ticks)
    e1.record(bench.stream)
    bench.barrier()
    ms = e0.elapsed_time(e1)
    n = int(ro.tick.item()) - done0
    s = ro.summary()
    tmax, = bench.max_over_ranks([ms])
    return {"workload": f"config5: closed-loop warm-started rollouts, {B} robots per GPU x {n} ticks, mu sweep 0.3-1.0, "
                        "SRBD plant (DART unavailable), CUDA graph of 10 ticks",
            "value": B * world * n / (tmax * 1e-3), "unit": "robot-ticks/s", "scaling": "weak",
            "ms_per_tick": tmax / max(n, 1), "ticks": n, "mean_iters": s["mean_iters"], "unsolved": s["unsolved"],
            "cache_hit_frac": s["cache_hit_frac"], "rms_pos_err_m": s["rms_pos_err"], "finite": s["finite"],
            "graph_replays_count_as_launches": int(ro.mpc.launch_count - l0)}


def run_ours(args):
    import torch
    import torch.distributed as dist
    import mpc_b200 as pkg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    bench = Bench(torch, dist, dev, world)
    B, N = args.batch, args.horizon
    gaits = tuple(args.gaits.split(","))
    # every rank draws its own shard of the global batch (batch-index sharding, no exchange)
    pb = pkg.problems.synthetic_batch(B, N=N, gaits=gaits, seed=rank)
    host = pb.f32()
    pinned = [torch.from_numpy(a).pin_memory() for a in host]
    dargs = [t.to(dev) for t in pinned]
    mpc = pkg.BatchedMPC(N=N, max_batch=B, device=local, warm_mode=0)
    out = mpc.alloc_outputs(B, want_X=True, device=dev)
    stream = bench.stream
    for _ in range(max(args.warmup, 3)):
        mpc.solve(*dargs, out=out)
    bench.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = mpc.launch_count
    # --- kernel-resident timing: inputs already in HBM, per-step CUDA events, L2 flushed ----
    t_wall0 = time.perf_counter()
    step_ms = bench.timed_steps(lambda: mpc.solve(*dargs, out=out), args.steps, warmup=0)
    t_wall = time.perf_counter() - t_wall0
    launches = mpc.launch_count - l0
    dev_ms = sum(step_ms)
    iters = out[2].cpu().numpy()
    status = out[5].cpu().numpy()
    if args.dump_outputs and rank == 0:       # before kernel_times() solves into the same buffers again
        dump_outputs(args.dump_outputs, U=out[0], X=out[1], iters=out[2], pri_res=out[3], dua_res=out[4],
                     status=out[5])

    kern_ms = kernel_times(pkg, bench, N, B, local, dargs, out, args.steps)

    # --- warm start (SURVEY.md 8d, config 2): x of the same problems one tick earlier, y = 0 (the
    # reference's semantics, src/mpc.py:270-271).  The previous-tick solve and the restore of the
    # warm state are outside the timed events; only the warm-started solve is timed.
    pb_prev = pkg.problems.synthetic_batch(B, N=N, gaits=gaits, seed=rank, tick_shift=-1)
    prev_args = [torch.from_numpy(a).to(dev) for a in pb_prev.f32()]
    mpc_w = pkg.BatchedMPC(N=N, max_batch=B, device=local, warm_mode=1)
    out_prev = mpc_w.alloc_outputs(B, want_X=False, device=dev)
    out_w = mpc_w.alloc_outputs(B, want_X=True, device=dev)
    mpc_w.solve(*prev_args, want_X=False, out=out_prev)
    x_prev = out_prev[0].clone()
    warm_ms = []
    for i in range(args.steps + 3):
        mpc_w.set_warm(x_prev)
        bench.flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        mpc_w.solve(*dargs, out=out_w)
        e1.record(stream)
        e1.synchronize()
        if i >= 3:
            warm_ms.append(e0.elapsed_time(e1))
    warm_iters = out_w[2].cpu().numpy()
    warm_status = out_w[5].cpu().numpy()
    bench.barrier()
    mpc_w.close()

    # --- end to end: host (pinned) buffers through cmpc_solve_host, copies inside the timing ----
    hin = [t.numpy() for t in pinned]
    pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()
    hout = (pin((B, N, 12), torch.float32), None, pin((B,), torch.int32),
            pin((B,), torch.float32), pin((B,), torch.float32), pin((B,), torch.int32))
    for _ in range(3):
        mpc.solve_host(*hin, want_X=False, out=hout)
    bench.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        mpc.solve_host(*hin, want_X=False, out=hout)
    torch.cuda.synchronize(dev)
    e2e_block_s = time.perf_counter() - t0
    bench.barrier()
    # the clocks were sampled through the device-timed steps, the warm-start pass and the blocking end-to-end loop;
    # the sampler stops here: on part of the boxes of this pool an nvidia-smi query loop running beside the
    # pipelined loop below costs it 25-35 % (0.30 instead of 0.23 ms per step, same box, same process)
    clocks = sampler.stop() if rank == 0 else None
    # the same steps double-buffered through cmpc_solve_host_async / cmpc_host_wait: step k+1 is submitted
    # (its own page-locked input and output buffers) before step k is waited for, so its host-to-device copies
    # and the host side of the call overlap the solve of step k; every step moves its inputs and results over PCIe
    # what this box's copy engines deliver on one step's inputs (the pipelined path is bound by it where it is
    # slower than the solve: boxes of the pool differ, 15-60 GB/s)
    dst = [torch.empty_like(t, device=dev) for t in pinned]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h2d_ms = []
    for _ in range(5):
        ev0.record()
        for d_, t_ in zip(dst, pinned):
            d_.copy_(t_, non_blocking=True)
        ev1.record()
        torch.cuda.synchronize(dev)
        h2d_ms.append(ev0.elapsed_time(ev1))
    h2d_gbs = sum(t.numel() * t.element_size() for t in pinned) / (statistics.median(h2d_ms) * 1e-3) / 1e9
    del dst
    d2h_src = torch.empty((B, N, 12), dtype=torch.float32, device=dev)       # one step's forces, the bulk of the results
    d2h_dst = torch.empty((B, N, 12), dtype=torch.float32).pin_memory()
    d2h_ms = []
    for _ in range(5):
        ev0.record()
        d2h_dst.copy_(d2h_src, non_blocking=True)
        ev1.record()
        torch.cuda.synchronize(dev)
        d2h_ms.append(ev0.elapsed_time(ev1))
    d2h_gbs = d2h_src.numel() * 4 / (statistics.median(d2h_ms) * 1e-3) / 1e9
    del d2h_src, d2h_dst
    bufs = [(hin, hout)]
    for _ in range(2):        # three buffer sets: the host runs up to two submissions ahead of the wait
        bufs.append(([torch.from_numpy(a).clone().pin_memory().numpy() for a in hin],
                     (pin((B, N, 12), torch.float32), None, pin((B,), torch.int32),
                      pin((B,), torch.float32), pin((B,), torch.float32), pin((B,), torch.int32))))
    e2e_s, reps, submit_us = e2e_block_s, [], [0.0]
    if int(mpc.cfg.host_zero_copy):
        for k in range(3):
            mpc.host_wait(mpc.solve_host_async(*bufs[k][0], out=bufs[k][1]))
        submit_us = []
        # the K-step loop lasts a few ms: one nvidia-smi sample (every 100 ms, driver lock) inside it costs up to 30 %,
        # and the first repetitions after the blocking loop run up to 40 % slower on part of the boxes (transient
        # of ~50 ms).  Steady state: ~1500 steps in repetitions of K (5 at least, 40 at most; the same count on
        # every rank), median.
        for _ in range(max(5, min(40, 1500 // max(args.steps, 1)))):
            bench.barrier()
            t0 = time.perf_counter()
            tickets = []
            for k in range(args.steps):
                h0 = time.perf_counter()
                tickets.append(mpc.solve_host_async(*bufs[k % 3][0], out=bufs[k % 3][1]))
                submit_us.append((time.perf_counter() - h0) * 1e6)
                if k >= 2:
                    mpc.host_wait(tickets[k - 2])
            for tk in tickets[-2:]:
                mpc.host_wait(tk)
            reps.append(time.perf_counter() - t0)
        e2e_s = statistics.median(reps)
        for q in bufs[1:]:
            assert np.array_equal(hout[0], q[1][0]) and np.array_equal(hout[2], q[1][2])
        bench.barrier()

    # --- latency: B=1 end-to-end p50, batch wall p50 ----------------------------------------
    lat = {}
    if rank == 0:
        one = [t[:1].contiguous() for t in dargs]
        out1 = mpc.alloc_outputs(1, want_X=True, device=dev)
        ts = []
        for i in range(220):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            mpc.solve(*one, out=out1)
            e1.record(stream)
            e1.synchronize()
            if i >= 20:
                ts.append(e0.elapsed_time(e1))
        lat = {"b1_solve_p50_us": 1e3 * statistics.median(ts),
               "batch_p50_ms": statistics.median(step_ms),
               "batch_amortised_p50_us_per_solve": 1e3 * statistics.median(step_ms) / B}

    # --- reduce over ranks: max time ------------------------------------------------------------
    dev_ms_max, e2e_s_max, warm_ms_max, e2e_block_s_max = bench.max_over_ranks([dev_ms, e2e_s, sum(warm_ms), e2e_block_s])
    ranks = per_rank_block(bench, kern_ms, step_ms, iters)

    try:
        fp32_peak = pkg._capi.fp32_peak(local) * 1e12
        fp32_src = "measured in this run (cmpc_fp32_peak: 8-chain FMA kernel, best of 4)"
    except Exception:
        fp32_peak = 148 * 128 * 2 * 1.965e9
        fp32_src = "148 SM x 128 lanes x 2 x 1.965 GHz (nominal)"

    # --- the other BASELINE configs and the sharded-identity check (all ranks take part) ----------
    configs = {}
    shard = None
    if not args.no_configs:
        P = pkg.problems
        lo, hi = pkg.sharding.shard_range(65536, rank, world)
        pb3 = P.synthetic_batch(65536, N=10, gaits=P.GAIT_NAMES, seed=0, mu=(0.3, 1.0)).slice(lo, hi)
        configs["config3"] = run_config(
            pkg, bench, torch, local, rank, world,
            f"config3: ONE global batch of 65536 mixed-gait problems (trot/pronk/amble/pseudo-gallop, mu 0.3-1.0), "
            f"N=10, contiguous batch-index shards over {world} GPU(s), cold start",
            pb3, max(args.steps // 3, 5), fp32_peak, "strong", global_batch=65536)
        del pb3
        pb4 = P.synthetic_batch(16384, N=30, gaits=("trot",), seed=rank)
        configs["config4"] = run_config(
            pkg, bench, torch, local, rank, world,
            "config4: long horizon N=30 trot, 16384 problems per GPU, cold start",
            pb4, max(args.steps // 6, 3), fp32_peak, "weak")
        pb4_cpu = pb4.slice(0, 256)
        del pb4
        configs["config5"] = run_rollout(pkg, bench, torch, local, world, args.rollout_ticks)
        shard = sharding_check(pkg, bench, torch, dist, local, rank, world)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    total = B * world * args.steps
    value = total / (dev_ms_max * 1e-3)
    e2e_val = total / e2e_s_max
    hbm_peak, peak_src = measured_peaks()
    flops, smem_b, hbm_b = algorithmic_work(N, pb.stance.sum((1, 2)), iters)
    kern_s = statistics.mean(kern_ms) * 1e-3         # this rank's mean solve-kernel launch duration
    ach_gbs = hbm_b * B / kern_s / 1e9
    # DRAM traffic and the shared-memory pipe share come from the committed ncu capture; they are
    # quoted only while the kernel source is the one that was profiled
    traffic, ncu_note, smem_pipe_pct = None, "no ncu capture on record", None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp) and (B, N, gaits) == (BATCH, HORIZON, ("trot",)):
        tj = json.load(open(tp))
        if tj.get("kernel_source_sha") in (None, kernel_source_sha()):
            traffic = tj.get("solve_kernel_dram_bytes_per_launch")
            smem_pipe_pct = tj.get("smem_pipe_pct_of_peak")
            ncu_note = tj.get("source", "profiles/traffic.json")
        else:
            ncu_note = "profiles/traffic.json was captured on an older kernel source: not quoted"
    smem_peak = 148 * 128 * 1.965e9
    fr_fp32 = flops * B / kern_s / fp32_peak
    fr_smem = smem_b * B / kern_s / smem_peak
    fr_hbm = ach_gbs / hbm_peak
    kname = f"cmpc::solve_kernel<{N},...> (dense" + (", tensor-core sweep)" if N == 10 else ")") if N <= 16 else f"cmpc::solve_riccati_kernel<{N},...> (stage-wise)"
    # SURVEY.md 8(d): the roofline fraction is the LARGEST of the three (FP32 pipe, shared memory, HBM)
    binding = max((fr_fp32, "fp32"), (fr_hbm, "hbm"))
    roof = {"bound": binding[1],
            "achieved": flops * B / kern_s / 1e12 if binding[1] == "fp32" else ach_gbs,
            "peak": fp32_peak / 1e12 if binding[1] == "fp32" else hbm_peak,
            "unit": "TFLOP/s" if binding[1] == "fp32" else "GB/s",
            "frac": binding[0], "traffic": traffic, "traffic_source": ncu_note,
            "peak_source": fp32_src if binding[1] == "fp32" else peak_src,
            "kernel": kname, "kernel_ms": statistics.mean(kern_ms),
            "kernel_share_of_step": statistics.mean(kern_ms) / (dev_ms / args.steps),
            "timing": "cudaEvent pair recorded by libcmpc on the launching stream around the solve kernel only "
                      "(cfg.time_kernel), mean over the timed steps of a second pass with the same inputs",
            "note": "on-chip bound path (SURVEY.md 8d): the binding roof is the FP32 FMA pipe with the survey's "
                    "algorithmic FLOP model; the HBM and shared-memory fractions are listed beside it",
            "fp32": {"algorithmic_flop_per_solve": flops, "achieved_tflops": flops * B / kern_s / 1e12,
                     "peak_tflops": fp32_peak / 1e12, "frac": fr_fp32, "peak_source": fp32_src},
            "hbm": {"algorithmic_bytes_per_solve": hbm_b, "achieved_gbs": ach_gbs, "peak_gbs": hbm_peak,
                    "frac": fr_hbm, "peak_source": peak_src},
            "smem": {"model_bytes_per_solve": smem_b, "model_frac_of_nominal_37TBs": fr_smem,
                     "ncu_smem_pipe_pct_of_peak": smem_pipe_pct,
                     "note": "the survey's 4Kn^2-byte model is of a triangular-solve algorithm this kernel does "
                             "not run; the ncu figure is the measured shared-memory pipe utilisation"}}
    in_bytes = sum(a.nbytes for a in host)
    out_bytes = sum(a.nbytes for a in hout if a is not None)
    line = {
        "metric": "QP solves/sec", "value": value, "unit": "solves/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms_max / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD if (B, N, gaits) == (BATCH, HORIZON, ("trot",)) else
                   f"batch {B} x N={N} gaits={','.join(gaits)} per GPU, cold start",
                   "batch_per_gpu": B, "horizon": N, "gaits": list(gaits), "sharding": f"batch-index x{world}",
                   "l2": "flushed between steps (256 MiB fill), per-step CUDA-event timing",
                   "solver": {"rho": float(mpc.cfg.rho), "sigma": float(mpc.cfg.sigma),
                              "alpha": float(mpc.cfg.alpha), "eps_abs": float(mpc.cfg.eps_abs),
                              "eps_rel": float(mpc.cfg.eps_rel), "check_every": int(mpc.cfg.check_every)},
                   "mean_iters": float(iters.mean()), "max_iters": int(iters.max()),
                   "solved_frac": float((status == 1).mean())},
        "roofline": roof,
        "e2e": {"value": e2e_val, "unit": "solves/s", "h2d_bytes_per_step": in_bytes,
                "d2h_bytes_per_step": out_bytes,
                "blocking_value": total / e2e_block_s_max,
                "rank0_ms_per_step_of_the_repetitions": [round(r_ / args.steps * 1e3, 4) for r_ in reps],
                "rank0_h2d_copy_engine_gbs": h2d_gbs, "rank0_d2h_copy_engine_gbs": d2h_gbs,
                "note": "may exceed `value`: the device-resident steps are timed one by one with the L2 flushed in between, "
                        "the pipelined steps run back to back on inputs the copy engines have just delivered",
                "rank0_host_us_per_submission": {"p50": float(np.percentile(submit_us, 50)), "p95": float(np.percentile(submit_us, 95)),
                                                 "max": float(np.max(submit_us))},
                "api": ("cmpc_solve_host_async + cmpc_host_wait, up to three steps in flight, each with its own page-locked "
                        "input and output buffers: the inputs of step k+1 are copied by the copy engines "
                        "(cudaMemcpyAsync) into a device arena while step k is solved and the results of step k are copied "
                        "back while step k+1 is solved (median over ~1500 steps in repetitions of the K steps); blocking_value = the same "
                        "steps through the blocking cmpc_solve_host (kernel reads / writes host memory in place)"
                        if int(mpc.cfg.host_zero_copy) else "cmpc_solve_host, staged with chunked cudaMemcpyAsync")},
        "warm_start": {"value": total / (warm_ms_max * 1e-3), "unit": "solves/s",
                       "ms_per_step": warm_ms_max / args.steps, "mean_iters": float(warm_iters.mean()),
                       "max_iters": int(warm_iters.max()), "solved_frac": float((warm_status == 1).mean()),
                       "what": "same batch warm-started with the forces of the same problems one tick earlier "
                               "(x unshifted, y = 0: the reference's set_initial semantics), L2 flushed, CUDA events"},
        "per_rank": ranks,
        "configs": configs,
        "sharding_check": shard,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "latency": lat,
        "wall_s_timed_region": t_wall,
    }
    if not args.no_cpu_baseline and world == 1:
        try:
            from oracle import cpu_baseline
            sample = args.cpu_sample or B
            info = cpu_baseline.solve_batch(pb.slice(0, sample))
            line["cpu_baseline"] = {
                "value": sample / info["seconds"], "unit": "solves/s", "cores": info["threads"],
                "kind": info["kind"],
                "sample": (f"the full batch of {B} problems" if sample == B else f"first {sample} of the {B} problems")
                          + f", {info['threads']} host threads, mean {info['mean_iters']:.1f} OSQP iterations"}
            if not args.no_configs:
                i4 = cpu_baseline.solve_batch(pb4_cpu)
                line["cpu_baseline"]["config4_n30"] = {
                    "value": pb4_cpu.B / i4["seconds"], "unit": "solves/s", "cores": i4["threads"],
                    "sample": f"first {pb4_cpu.B} of the 16384 N=30 problems, mean {i4['mean_iters']:.1f} OSQP iterations"}
        except Exception as exc:      # the oracle is a checker; a missing build must not kill the bench
            line["cpu_baseline"] = {"value": None, "unit": "solves/s", "cores": 0, "kind": "port",
                                    "sample": f"unavailable: {exc}"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
