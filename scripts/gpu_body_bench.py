"""Cost of per-robot bodies (cmpc_set_body) on one GPU, in one process.

config 2 (4096 trot problems, N = 10, cold start) and config 4 (16384 trot problems, N = 30, cold start): the
solve kernel alone (cfg.time_kernel) and the whole cmpc_solve step (CUDA events), L2 flushed (256 MiB fill)
before every step, for three handles in alternation: one that never received a body (the kernels bench.py
runs), one with random_bodies, one with the configuration's body set explicitly (the body kernels on the
same arithmetic as the first).  config 5 (8192 robots x 1000 ticks, graph replay of 10 ticks) with and
without random bodies.  Prints the GPU name and power limit with the numbers, one JSON line per result.

    python scripts/gpu_body_bench.py [--steps 30] [--ticks 1000]
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
from mpc_b200.problems import synthetic_batch, random_bodies  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def make_handles(N, B):
    dev = torch.device("cuda", 0)
    f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    arms = {}
    for name in ("no_body", "random_bodies", "config_body"):
        h = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0, time_kernel=1)
        if name == "random_bodies":
            m, ib = random_bodies(B, seed=0)
            h.set_body(f32(m), f32(ib))
        elif name == "config_body":
            h.set_body(f32(np.full(B, h.cfg.mass)), f32(np.tile(np.diag(np.array(h.cfg.ibody_inv[:])), (B, 1, 1))))
        arms[name] = h
    torch.cuda.synchronize()
    return arms


def solve_arms(label, N, B, steps, flush):
    pb = synthetic_batch(B, N=N, gaits=("trot",), seed=0)
    args = [torch.from_numpy(a).cuda() for a in pb.f32()]
    arms = make_handles(N, B)
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
    same = bool(torch.equal(outs["no_body"][0], outs["config_body"][0]))
    base = np.median(kern["no_body"])
    for k in arms:
        print(json.dumps({"workload": label, "arm": k, "kernel_ms_median": float(np.median(kern[k])),
                          "kernel_ms_min": float(np.min(kern[k])), "kernel_ms_max": float(np.max(kern[k])),
                          "step_ms_median": float(np.median(step[k])),
                          "solves_per_s_step": B / (float(np.median(step[k])) * 1e-3),
                          "kernel_vs_no_body": float(np.median(kern[k]) / base - 1.0),
                          "mean_iters": iters[k][0], "max_iters": iters[k][1], "steps": steps}))
    print(json.dumps({"workload": label, "config_body_U_equals_no_body_U": same}))


def rollout_arm(bodies, ticks):
    B = 8192
    kw = {}
    if bodies:
        kw["mass"], kw["ibody_inv"] = random_bodies(B, seed=0)
    ro = pkg.ClosedLoopRollout(B, N=10, gaits=("trot",), mu=(0.3, 1.0), seed=0, **kw)
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
    return {"workload": f"config5: {B} robots x {n} ticks, graph replay", "arm": "random_bodies" if bodies else "no_body",
            "ms_per_tick": e0.elapsed_time(e1) / max(n, 1), "mean_iters": s["mean_iters"], "unsolved": s["unsolved"],
            "cache_hit_frac": s["cache_hit_frac"], "com_z_min": s["com_z_min"], "com_z_max": s["com_z_max"],
            "finite": s["finite"]}


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
    for rep in range(2):                          # alternate the two rollout arms twice
        for bodies in (False, True):
            print(json.dumps(dict(rollout_arm(bodies, a.ticks), rep=rep)))
    print(json.dumps(gpu_info()))


if __name__ == "__main__":
    main()
