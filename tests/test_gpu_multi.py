"""Hardware multi-GPU identity (SURVEY.md section 4-iv / 8e): ONE global batch solved as contiguous
shards on 2 GPUs (one torchrun rank per GPU), gathered over NCCL with sharding.gather_results, must be
bit-identical to the single-GPU result of the whole batch.  Skipped on boxes with one GPU (bench.py
repeats the same check at every --gpus N and prints it in its JSON line)."""
import json
import os
import subprocess
import sys

import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import json, os, sys
sys.path.insert(0, %r)
import torch, torch.distributed as dist
import mpc_b200 as pkg
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
Bg, N = 3001, 10                                    # ragged shards
pb = pkg.problems.synthetic_batch(Bg, N=N, gaits=pkg.problems.GAIT_NAMES, seed=5, mu=(0.3, 1.0))
mpc = pkg.BatchedMPC(N=N, max_batch=Bg, device=local, warm_mode=0)
lo, hi, U, X, st = pkg.sharding.solve_sharded(mpc, pb, rank, world, device=dev)
u0, it, status = pkg.sharding.gather_results(U[:, 0, :].contiguous(), st.iters, st.status, Bg)
ok = None
if rank == 0:
    full = [torch.from_numpy(a).to(dev) for a in pb.f32()]
    Uf, _, sf = mpc.solve(*full)
    torch.cuda.synchronize()
    ok = dict(u0=bool(torch.equal(u0, Uf[:, 0, :])), iters=bool(torch.equal(it, sf.iters)),
              status=bool(torch.equal(status, sf.status)), world=world, shard=[lo, hi], solved=int((sf.status == 1).sum()))
    print("RESULT " + json.dumps(ok), flush=True)
dist.barrier()
dist.destroy_process_group()
''' % ROOT


def test_two_gpu_shards_equal_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29517", str(script)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    line = [l for l in res.stdout.splitlines() if l.startswith("RESULT ")][-1]
    ok = json.loads(line[len("RESULT "):])
    assert ok["u0"] and ok["iters"] and ok["status"] and ok["world"] == 2 and ok["solved"] == 3001


@pytest.mark.parametrize("N,B", [(40, 512), (10, 3072)])
def test_second_gpu_in_one_process_matches_the_first(N, B):
    """Handles on two GPUs in one process.  Function attributes and occupancy are per device, so the launch
    set-up must run on each device it launches on: N = 40 needs the Riccati kernel's dynamic shared-memory
    opt-in, and N = 10 at 3072 problems (1.5-4 waves) sizes its reserved-SM launch from the occupancy of the
    device.  Device 1 must compute bit for bit what device 0 computes, and leave the current device at 0."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import mpc_b200 as pkg
    torch.cuda.set_device(0)
    pb = pkg.problems.synthetic_batch(B, N=N, gaits=pkg.problems.GAIT_NAMES, seed=5, mu=(0.3, 1.0))
    outs = []
    for d in (0, 1):
        mpc = pkg.BatchedMPC(N=N, max_batch=B, device=d, warm_mode=0)
        U, X, st = mpc.solve(*[torch.from_numpy(a).to(torch.device("cuda", d)) for a in pb.f32()])
        torch.cuda.synchronize(d)
        assert torch.cuda.current_device() == 0
        outs.append([t.cpu() for t in (U, X, st.iters, st.pri_res, st.dua_res, st.status)])
        mpc.close()
    for a, b in zip(*outs):
        assert torch.equal(a, b)
