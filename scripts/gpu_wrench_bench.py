"""Cost of per-robot external wrenches (cmpc_set_wrench) on one GPU, in one process.

config 2 (4096 trot problems, N = 10, cold start) and config 4 (16384 trot problems, N = 30, cold start): the
solve kernel alone (cfg.time_kernel) and the whole cmpc_solve step (CUDA events), L2 flushed (256 MiB fill)
before every step, for three handles in alternation: one that never received a wrench (the kernels bench.py runs),
one with a zero wrench set explicitly (the same solve kernels plus the shift and finish passes) and one with
random_wrenches; mean and max ADMM iterations of each.  The shift and finish kernels are timed in a separate
torch.profiler pass of the random-wrench handle.  Then the time of one cmpc_set_wrench of the whole batch (after
the first call, which allocates), and config 5 (8192 closed-loop trotting robots, CUDA graph of 10 ticks) with and
without a constant 15 N lateral push.  Prints the GPU name and power limit with the numbers, one JSON line per
result.

    python scripts/gpu_wrench_bench.py [--steps 30] [--ticks 1000]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mpc_b200 as pkg  # noqa: E402
from mpc_b200.problems import synthetic_batch, random_wrenches  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def f32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def make_handles(N, B):
    rw = tuple(map(f32, random_wrenches(B, N, seed=0)))
    arms = {}
    for name in ("no_wrench", "zero_wrench", "random_wrenches"):
        h = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0, time_kernel=1)
        if name == "zero_wrench":
            h.set_wrench(f32(np.zeros((B, N, 3))), f32(np.zeros((B, N, 3))))
        elif name == "random_wrenches":
            h.set_wrench(*rw)
        arms[name] = h
    torch.cuda.synchronize()
    return arms, rw


def set_wrench_ms(h, rw, reps=50):
    """one cmpc_set_wrench of the whole batch (the handle has made its first call), CUDA events"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(5):
        h.set_wrench(*rw)
    e0.record()
    for _ in range(reps):
        h.set_wrench(*rw)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def pass_kernel_ms(h, args, out, flush, steps=10):
    """mean device time per solve of the wrench shift and finish kernels, from a torch.profiler pass of its own"""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            flush.fill_(1)
            h.solve(*args, out=out)
        torch.cuda.synchronize()
    res = {}
    for name in ("wrench_shift_kernel", "wrench_finish_kernel"):
        ev = [e for e in prof.key_averages() if name in e.key]
        us = sum(getattr(e, "device_time_total", 0.0) for e in ev)
        n = sum(e.count for e in ev)
        res[name + "_ms_mean"] = us / n / 1e3 if n else None
    return res


def solve_arms(label, N, B, steps, flush):
    pb = synthetic_batch(B, N=N, gaits=("trot",), seed=0)
    args = [torch.from_numpy(a).cuda() for a in pb.f32()]
    arms, rw = make_handles(N, B)
    outs = {k: h.alloc_outputs(B) for k, h in arms.items()}
    kern = {k: [] for k in arms}
    step = {k: [] for k in arms}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(steps + 3):
        for k, h in arms.items():                 # alternate the arms step by step
            flush.fill_(1)
            e0.record()
            h.solve(*args, out=outs[k])
            e1.record()
            e1.synchronize()
            if i >= 3:
                kern[k].append(h.last_kernel_ms)
                step[k].append(e0.elapsed_time(e1))
    same = all(torch.equal(a, b) for a, b in zip(outs["no_wrench"], outs["zero_wrench"]))
    base_k, base_s = np.median(kern["no_wrench"]), np.median(step["no_wrench"])
    for k in arms:
        it = outs[k][2].float()
        print(json.dumps({"workload": label, "arm": k, "kernel_ms_median": float(np.median(kern[k])),
                          "kernel_ms_min": float(np.min(kern[k])), "kernel_ms_max": float(np.max(kern[k])),
                          "step_ms_median": float(np.median(step[k])),
                          "solves_per_s_step": B / (float(np.median(step[k])) * 1e-3),
                          "kernel_vs_no_wrench": float(np.median(kern[k]) / base_k - 1.0),
                          "step_vs_no_wrench": float(np.median(step[k]) / base_s - 1.0),
                          "mean_iters": float(it.mean()), "max_iters": int(it.max()), "steps": steps}))
    print(json.dumps({"workload": label, "zero_wrench_outputs_equal_no_wrench": same,
                      "set_wrench_ms": set_wrench_ms(arms["random_wrenches"], rw),
                      **pass_kernel_ms(arms["random_wrenches"], args, outs["random_wrenches"], flush)}))


def rollout(ticks, push):
    B = 8192
    force = np.tile([0.0, 15.0, 0.0], (B, 1)) if push else None
    ro = pkg.ClosedLoopRollout(B, N=10, gaits=("trot",), mu=(0.3, 1.0), seed=0, force=force)
    ro.capture(10)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = int(ro.tick.item())
    e0.record()
    ro.run(ticks)
    e1.record()
    e1.synchronize()
    n = int(ro.tick.item()) - t0
    s = ro.summary()
    return {"workload": f"config5: {B} closed-loop trotting robots x {n} ticks, CUDA graph of 10 ticks",
            "arm": "15 N lateral push" if push else "no wrench", "ms_per_tick": e0.elapsed_time(e1) / max(n, 1),
            "mean_iters": s["mean_iters"], "unsolved": s["unsolved"], "cache_hit_frac": s["cache_hit_frac"],
            "rms_pos_err_m": s["rms_pos_err"], "finite": s["finite"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--ticks", type=int, default=1000)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    print(json.dumps(gpu_info()))
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    solve_arms("config2: 4096 trot, N=10, cold", 10, 4096, a.steps, flush)
    solve_arms("config4: 16384 trot, N=30, cold", 30, 16384, max(a.steps // 3, 5), flush)
    for push in (False, True, False, True):       # alternated
        print(json.dumps(rollout(a.ticks, push)))
    print(json.dumps(gpu_info()))


if __name__ == "__main__":
    main()
