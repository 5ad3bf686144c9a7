"""Small run of every kernel for compute-sanitizer --tool memcheck (one tool per gpurun call)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import mpc_b200 as pkg
from mpc_b200.problems import synthetic_batch, GAIT_NAMES
for N, B, variants in ((10, 48, (0, 5)), (5, 8, (0,)), (20, 8, (0, 5)), (30, 6, (0, 5)), (40, 2, (0,)), (60, 2, (0,))):
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=1)
    args = [torch.from_numpy(a).cuda() for a in pb.f32()]
    for v in variants:
        mpc = pkg.BatchedMPC(N=N, max_batch=B, kernel_variant=v, lpt_schedule=4, max_iter=60)
        U, X, st = mpc.solve(*args)
        torch.cuda.synchronize()
        print(N, v, "iters", st.iters.float().mean().item(), flush=True)
    if N <= 30:
        H, g = mpc.condense(*args[:4]); torch.cuda.synchronize()
pb = synthetic_batch(64, N=10, seed=2)
hin = [torch.from_numpy(a).pin_memory().numpy() for a in pb.f32()]
mpc = pkg.BatchedMPC(N=10, max_batch=64, lpt_schedule=4)
print("host zero-copy", mpc.solve_host(*hin)[2].iters.mean())
print("host staged", mpc.solve_host(*pb.f32())[2].iters.mean())
ro = pkg.ClosedLoopRollout(32, N=10, gaits=("trot",), mu=(0.3, 1.0), seed=0)
ro.run(5, use_graph=False)
torch.cuda.synchronize()
print("rollout ok", ro.summary()["finite"])
