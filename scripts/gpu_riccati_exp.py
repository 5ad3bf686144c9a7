"""GPU experiment (round 2): stage-wise (Riccati) kernel against the dense kernel per horizon:
cold-start solves/s and agreement of the results on the same batch.  Riccati = default for N >= 20 and
kernel_variant 5 for N <= 16; dense = the other one."""
import json, sys, os
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mpc_b200 as pkg
from mpc_b200.problems import synthetic_batch, GAIT_NAMES

def run(pb, variant, reps=5, **opts):
    dev = torch.device("cuda", 0)
    args = [torch.from_numpy(a).to(dev) for a in pb.f32()]
    mpc = pkg.BatchedMPC(N=pb.N, max_batch=pb.B, warm_mode=0, time_kernel=1, kernel_variant=variant, **opts)
    out = mpc.alloc_outputs(pb.B)
    ms = []
    for i in range(reps + 2):
        mpc.solve(*args, out=out)
        torch.cuda.synchronize()
        if i >= 2:
            ms.append(mpc.last_kernel_ms)
    res = dict(ms=float(np.median(ms)), U=out[0].cpu().numpy(), X=out[1].cpu().numpy(), it=out[2].cpu().numpy(), st=out[5].cpu().numpy())
    mpc.close()
    return res

if __name__ == "__main__":
    for N, B, gaits in ((10, 4096, ("trot",)), (20, 4096, ("trot",)), (30, 16384, ("trot",))):
        pb = synthetic_batch(B, N=N, gaits=gaits, seed=0)
        a = run(pb, 0 if N <= 16 else 5)      # dense
        r = run(pb, 5 if N <= 16 else 0)      # Riccati
        same = (a["st"] == 1) & (r["st"] == 1)
        print(json.dumps(dict(N=N, B=B, dense_ms=a["ms"], dense_solves_s=B / a["ms"] * 1e3, ric_ms=r["ms"], ric_solves_s=B / r["ms"] * 1e3,
                              speedup=a["ms"] / r["ms"], dense_iters=float(a["it"].mean()), ric_iters=float(r["it"].mean()),
                              ric_solved=float((r["st"] == 1).mean()), dense_solved=float((a["st"] == 1).mean()),
                              max_dX=float(np.abs(a["X"][same] - r["X"][same]).max()), iters_equal_frac=float((a["it"] == r["it"]).mean()))), flush=True)
