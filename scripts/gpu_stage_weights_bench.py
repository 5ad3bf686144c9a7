"""Cost of per-robot stage weights (cmpc_set_stage_weights) on one GPU, in one process.

config 2 (4096 trot problems, N = 10, cold start), config 4 (16384 trot problems, N = 30, cold start) and 4096 trot
problems at N = 60 (the per-stage weight loads of the Riccati sweeps): the solve kernel alone (cfg.time_kernel), L2
flushed (256 MiB fill) before every step, for four handles in alternation: one given the configuration's weights (the
BODY + WEIGHTS twins), one given zero-weight force references (the FORCE twins, which the STAGE kernels extend), one
given the configuration's weights on every stage (the STAGE kernels on the same arithmetic) and one with
random_stage_weights.  For each: mean and max ADMM iterations and the SOLVED rate; whether the uniform-stage arm
returns the same U as the FORCE twin.  Then the time of one cmpc_set_stage_weights call for the whole batch after the
first call, and of the first call (allocation and host-synchronous initialisation of every slot, the weight and
reference storage included).  Prints the GPU name and power limit with the numbers, one JSON line per result.

    python scripts/gpu_stage_weights_bench.py [--steps 30]
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
from mpc_b200.problems import synthetic_batch, random_stage_weights  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def f32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def make_handles(N, B):
    ws = f32(random_stage_weights(B, N, seed=0))
    arms, first_ms = {}, None
    for name in ("body_weights", "force_twin", "uniform_stage", "random_stage_weights"):
        h = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0, time_kernel=1)
        w = np.array(h.cfg.w[:])
        if name == "body_weights":
            h.set_weights(f32(np.tile(w, (B, 1))), f32(np.full(B, h.cfg.r_weight)))
        elif name == "force_twin":
            h.set_force_ref(f32(np.zeros((B, N, 4, 3))), f32(np.zeros((B, N, 4))))
        elif name == "uniform_stage":
            h.set_stage_weights(f32(np.tile(w, (B, N, 1))))
        else:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            h.set_stage_weights(ws)
            torch.cuda.synchronize()
            first_ms = (time.perf_counter() - t0) * 1e3
        arms[name] = h
    torch.cuda.synchronize()
    return arms, ws, first_ms


def set_stage_weights_ms(h, ws, reps=20):
    """one cmpc_set_stage_weights of the whole batch (the handle has made its first call), CUDA events"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        h.set_stage_weights(ws)
    e0.record()
    for _ in range(reps):
        h.set_stage_weights(ws)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def solve_arms(label, N, B, steps, flush):
    pb = synthetic_batch(B, N=N, gaits=("trot",), seed=0)
    args = [torch.from_numpy(a).cuda() for a in pb.f32()]
    arms, ws, first_ms = make_handles(N, B)
    outs = {k: h.alloc_outputs(B) for k, h in arms.items()}
    kern = {k: [] for k in arms}
    for i in range(steps + 3):
        for k, h in arms.items():                 # alternate the arms step by step
            flush.fill_(1)
            h.solve(*args, out=outs[k])
            torch.cuda.synchronize()
            if i >= 3:
                kern[k].append(h.last_kernel_ms)
    twin, ftwin = np.median(kern["body_weights"]), np.median(kern["force_twin"])
    for k in arms:
        it, st = outs[k][2], outs[k][5]
        print(json.dumps({"workload": label, "arm": k, "kernel_ms_median": float(np.median(kern[k])),
                          "kernel_ms_min": float(np.min(kern[k])), "kernel_ms_max": float(np.max(kern[k])),
                          "kernel_vs_body_weights": float(np.median(kern[k]) / twin - 1.0),
                          "kernel_vs_force_twin": float(np.median(kern[k]) / ftwin - 1.0),
                          "mean_iters": float(it.float().mean()), "max_iters": int(it.max()),
                          "solved_rate": float((st == 1).float().mean()), "steps": steps}))
    print(json.dumps({"workload": label,
                      "uniform_stage_U_equals_force_twin_U": bool(torch.equal(outs["force_twin"][0],
                                                                              outs["uniform_stage"][0])),
                      "set_stage_weights_ms": set_stage_weights_ms(arms["random_stage_weights"], ws),
                      "first_set_stage_weights_ms": first_ms}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    print(json.dumps(gpu_info()))
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    solve_arms("config2: 4096 trot, N=10, cold", 10, 4096, a.steps, flush)
    solve_arms("config4: 16384 trot, N=30, cold", 30, 16384, max(a.steps // 3, 5), flush)
    solve_arms("4096 trot, N=60, cold", 60, 4096, max(a.steps // 3, 5), flush)
    print(json.dumps(gpu_info()))


if __name__ == "__main__":
    main()
