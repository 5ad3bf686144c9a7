"""Cost of per-robot cost weights (cmpc_set_weights) on one GPU, in one process.

config 2 (4096 trot problems, N = 10, cold start) and config 4 (16384 trot problems, N = 30, cold start): the
solve kernel alone (cfg.time_kernel) and the whole cmpc_solve step (CUDA events), L2 flushed (256 MiB fill)
before every step, for four handles in alternation: one that never received weights (the kernels bench.py runs),
one given the configuration's body (the BODY twins, which the WEIGHTS twins extend), one given the configuration's
weights explicitly (the WEIGHTS twins on the same arithmetic as the first) and one with random_weights; mean and
max ADMM iterations of each, and whether the configuration-weights arm returns the same U as the first.  Then the
time of one cmpc_set_weights call for the whole batch at each size after the first call, and of the first call
(allocation and host-synchronous initialisation of every slot).  Prints the GPU name and power limit with the
numbers, one JSON line per result.

    python scripts/gpu_weights_bench.py [--steps 30]
"""

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mpc_b200 as pkg  # noqa: E402
from mpc_b200.problems import synthetic_batch, random_weights  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def f32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def make_handles(N, B):
    rw = tuple(map(f32, random_weights(B, seed=0)))
    arms, first_ms = {}, None
    for name in ("no_weights", "config_body", "config_weights", "random_weights"):
        h = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0, time_kernel=1)
        if name == "config_body":
            h.set_body(f32(np.full(B, h.cfg.mass)), f32(np.tile(np.array(h.cfg.ibody_inv[:]), (B, 1))).diag_embed())
        elif name == "config_weights":
            h.set_weights(f32(np.tile(np.array(h.cfg.w[:]), (B, 1))), f32(np.full(B, h.cfg.r_weight)))
        elif name == "random_weights":
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            h.set_weights(*rw)
            torch.cuda.synchronize()
            first_ms = (time.perf_counter() - t0) * 1e3
        arms[name] = h
    torch.cuda.synchronize()
    return arms, rw, first_ms


def set_weights_ms(h, rw, reps=20):
    """one cmpc_set_weights of the whole batch (the handle has made its first call), CUDA events"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        h.set_weights(*rw)
    e0.record()
    for _ in range(reps):
        h.set_weights(*rw)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def solve_arms(label, N, B, steps, flush):
    pb = synthetic_batch(B, N=N, gaits=("trot",), seed=0)
    args = [torch.from_numpy(a).cuda() for a in pb.f32()]
    arms, rw, first_ms = make_handles(N, B)
    outs = {k: h.alloc_outputs(B) for k, h in arms.items()}
    kern = {k: [] for k in arms}
    step = {k: [] for k in arms}
    iters = {}
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
    for k in arms:
        iters[k] = (float(outs[k][2].float().mean()), int(outs[k][2].max()))
    same = bool(torch.equal(outs["no_weights"][0], outs["config_weights"][0]))
    base, body = np.median(kern["no_weights"]), np.median(kern["config_body"])
    for k in arms:
        print(json.dumps({"workload": label, "arm": k, "kernel_ms_median": float(np.median(kern[k])),
                          "kernel_ms_min": float(np.min(kern[k])), "kernel_ms_max": float(np.max(kern[k])),
                          "step_ms_median": float(np.median(step[k])),
                          "solves_per_s_step": B / (float(np.median(step[k])) * 1e-3),
                          "kernel_vs_no_weights": float(np.median(kern[k]) / base - 1.0),
                          "kernel_vs_config_body": float(np.median(kern[k]) / body - 1.0),
                          "mean_iters": iters[k][0], "max_iters": iters[k][1], "steps": steps}))
    print(json.dumps({"workload": label, "config_weights_U_equals_no_weights_U": same,
                      "set_weights_ms": set_weights_ms(arms["random_weights"], rw),
                      "first_set_weights_ms": first_ms}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    print(json.dumps(gpu_info()))
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    solve_arms("config2: 4096 trot, N=10, cold", 10, 4096, a.steps, flush)
    solve_arms("config4: 16384 trot, N=30, cold", 30, 16384, max(a.steps // 3, 5), flush)
    print(json.dumps(gpu_info()))


if __name__ == "__main__":
    main()
