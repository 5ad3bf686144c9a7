"""Per-robot external wrench (cmpc_set_wrench) on the GPU: a zero wrench against no wrench, iterate parity and
converged solves against the fp64 oracle under the same wrench, slot ownership, host paths, the factorisation cache,
invalid wrenches, graph capture, condense, the plant against the model's prediction and the closed loop."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import mpc_b200 as pkg                                                      # noqa: E402
from mpc_b200 import _capi                                                  # noqa: E402
from mpc_b200.problems import (synthetic_batch, random_bodies, random_contacts, random_weights,  # noqa: E402
                               random_wrenches, DT, GAIT_NAMES)
from oracle import condensed_admm as ca, srbd_qp, tight_ipm as ipm         # noqa: E402
import body_oracle as bo                                                    # noqa: E402
import wrench_oracle as wo                                                  # noqa: E402

ATOL, RTOL = 1e-2, 1e-3
dev = torch.device("cuda", 0)


def f32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)


def r32(a):
    """what the device holds, in fp64 for the oracle"""
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def wrenches(B, N, seed):
    return tuple(r32(a) for a in random_wrenches(B, N, seed=seed))


def run(mpc, pb, slot0=0):
    U, X, st = mpc.solve(*[a.to(dev) for a in map(torch.from_numpy, pb.f32())], slot0=slot0)
    torch.cuda.synchronize()
    return U, X, st


def to_np(U, X, st):
    return dict(U=U.cpu().numpy().astype(np.float64), X=X.cpu().numpy().astype(np.float64),
                iters=st.iters.cpu().numpy(), status=st.status.cpu().numpy(),
                pri=st.pri_res.cpu().numpy(), dua=st.dua_res.cpu().numpy())


KEYS = ("U", "X", "iters", "status", "pri", "dua")


def same(a, b, sel=slice(None)):
    return all(np.array_equal(a[k][sel], b[k][sel], equal_nan=True) for k in KEYS)


@pytest.mark.parametrize("N,B,variant,cache,extra", [(10, 2048, 0, 0, 0), (10, 256, 0, 1, 0), (12, 64, 0, 0, 0),
                                                     (30, 64, 0, 0, 0), (30, 64, 0, 1, 0), (60, 16, 0, 0, 0),
                                                     (7, 64, 0, 0, 0), (10, 64, 5, 0, 0), (20, 64, 5, 0, 0),
                                                     (30, 64, 5, 0, 0), (10, 256, 0, 0, 1), (30, 64, 0, 1, 1),
                                                     (7, 64, 0, 0, 1), (60, 16, 0, 0, 1)])
def test_zero_wrench_is_bit_identical_to_no_wrench(N, B, variant, cache, extra):
    """An explicitly set zero wrench reproduces the handle without one bit for bit (the same solve kernels on a copy of
    x_des, and X untouched).  At N = 10 with 2048 problems the hardest-first order and the reserved-SM launch are
    active; `extra` gives both handles random bodies, contacts and weights."""
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=17)
    opts = dict(kernel_variant=variant, cache_factorization=cache, warm_mode=0)
    a = pkg.BatchedMPC(N=N, max_batch=B, **opts)
    b = pkg.BatchedMPC(N=N, max_batch=B, **opts)
    if extra:
        m, ib = random_bodies(B, seed=5)
        c = [f32(x) for x in random_contacts(B, N, seed=5)]
        w, rw = random_weights(B, seed=5)
        for h in (a, b):
            h.set_body(f32(m), f32(ib))
            h.set_contact(*c)
            h.set_weights(f32(w), f32(rw))
    b.set_wrench(f32(np.zeros((B, N, 3))), f32(np.zeros((B, N, 3))))
    for _ in range(2 if cache else 1):                # with the cache: the fresh factorisation, then the reuse
        assert same(to_np(*run(a, pb)), to_np(*run(b, pb)))
    if cache:
        assert torch.equal(a.cache_meta(B), b.cache_meta(B))


@pytest.mark.parametrize("N,variant", [(4, 0), (5, 0), (8, 0), (10, 0), (12, 0), (16, 0), (20, 0), (30, 0), (40, 0),
                                       (60, 0), (7, 0), (25, 0), (10, 5), (20, 5), (30, 5)])
def test_iterate_parity_with_random_wrenches(N, variant):
    B, K = 6, (50 if N < 60 else 120)
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=3)
    force, torque = wrenches(B, N, seed=N)
    mpc = pkg.BatchedMPC(N=N, max_batch=B, max_iter=K, check_every=100000, eps_abs=0.0, eps_rel=0.0, warm_mode=0,
                         adaptive_rho_interval=0, kernel_variant=variant)
    mpc.set_wrench(f32(force), f32(torque))
    out = to_np(*run(mpc, pb))
    assert np.all(out["iters"] == K)
    for b in range(B):
        x0, r, stance, xd, mu = pb.problem(b)
        ref = wo.admm_solve(x0, r, stance, xd, mu, DT, force[b], torque[b], fixed_iters=K, rho=float(mpc.cfg.rho),
                            sigma=float(mpc.cfg.sigma), alpha=float(mpc.cfg.alpha))
        err = np.abs(out["U"][b] - ref["U"])
        tr = (3e-3 if N < 60 else 6e-3) * np.abs(ref["U"]).max()
        assert np.all(err <= 2 * ATOL + tr + RTOL * np.abs(ref["U"])), (b, err.max())
        assert np.all(np.abs(out["X"][b].T - ref["X"]) <= 2e-4 + 1e-3 * np.abs(ref["X"]))
        sw = np.repeat(pb.stance[b].reshape(-1) == 0, 3)
        assert np.all(out["U"][b].reshape(-1)[sw] == 0.0)


@pytest.mark.parametrize("N", [10, 30])
def test_converged_solves_with_random_wrenches(N):
    B = 24
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=12)
    force, torque = wrenches(B, N, seed=100 + N)
    mpc = pkg.BatchedMPC(N=N, max_batch=B)
    mpc.set_wrench(f32(force), f32(torque))
    out = to_np(*run(mpc, pb))
    assert np.mean(out["status"] == 1) >= 0.9
    for b in range(0, B, 3):
        if out["status"][b] != 1:
            continue
        x0, r, stance, xd, mu = pb.problem(b)
        tight = wo.ipm_solve(x0, r, stance, xd, mu, DT, force[b], torque[b])
        J = srbd_qp.objective(out["X"][b].T, xd)
        assert abs(J / tight["J"] - 1.0) < 2e-2, (b, J, tight["J"])


@pytest.mark.parametrize("N,B", [(10, 2048), (30, 256), (7, 256)])
def test_slot_wrenches_belong_to_their_slots(N, B):
    """Wrenches at slot0 = 300: every problem equals the same problem solved with its wrench on a fresh handle, and the
    slots never set solve as on a handle without wrenches."""
    s0 = 300
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=23)
    force, torque = wrenches(B, N, seed=23)
    mpc = pkg.BatchedMPC(N=N, max_batch=s0 + B, warm_mode=0)
    mpc.set_wrench(f32(force), f32(torque), slot0=s0)
    fresh = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0)
    fresh.set_wrench(f32(force), f32(torque))
    assert same(to_np(*run(mpc, pb, slot0=s0)), to_np(*run(fresh, pb)))
    rest = synthetic_batch(s0, N=N, gaits=GAIT_NAMES, seed=24)
    assert same(to_np(*run(mpc, rest)), to_np(*run(pkg.BatchedMPC(N=N, max_batch=s0, warm_mode=0), rest)))


def test_host_paths_use_the_slot_wrench():
    B, N = 2048, 10
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=8)
    force, torque = wrenches(B, N, seed=8)

    def handle(**kw):
        h = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0, **kw)
        h.set_wrench(f32(force), f32(torque))
        torch.cuda.synchronize()
        return h
    ref = to_np(*run(handle(), pb))
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    zeros = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory().numpy()

    def pinned_out():
        return (zeros((B, N, 12), torch.float32), zeros((B, N + 1, 13), torch.float32), zeros((B,), torch.int32),
                zeros((B,), torch.float32), zeros((B,), torch.float32), zeros((B,), torch.int32))

    def check(U, X, st):
        assert np.array_equal(U, ref["U"].astype(np.float32)) and np.array_equal(X, ref["X"].astype(np.float32))
        assert np.array_equal(st.iters, ref["iters"]) and np.array_equal(st.status, ref["status"])
    hin = [pin(a) for a in pb.f32()]
    check(*handle().solve_host(*hin, out=pinned_out()))                         # zero-copy
    check(*handle(host_zero_copy=0).solve_host(*hin, out=pinned_out()))         # two chunks, engine copies
    check(*handle().solve_host(*pb.f32()))                                      # pageable, staged
    h = handle()
    out = pinned_out()
    h.host_wait(h.solve_host_async(*hin, out=out))
    U, X, it, _, _, stt = out
    check(U, X, type("S", (), dict(iters=it, status=stt)))


def test_set_wrench_keeps_the_factorisation_cache():
    """A standing batch reuses its cached factors after set_wrench exactly as without it."""
    B = 256
    pb = synthetic_batch(B, N=10, gaits=GAIT_NAMES, seed=21)
    force, torque = wrenches(B, 10, seed=21)
    opts = dict(warm_mode=0, cache_factorization=1, cache_max_iter=1000)
    a, b = pkg.BatchedMPC(N=10, max_batch=B, **opts), pkg.BatchedMPC(N=10, max_batch=B, **opts)
    for h in (a, b):
        run(h, pb)
        run(h, pb)
    before = a.cache_meta(B).cpu().numpy()
    assert before[:, 2].mean() > 0.8                                   # entries are valid
    a.set_wrench(f32(force), f32(torque))
    torch.cuda.synchronize()
    assert np.array_equal(a.cache_meta(B).cpu().numpy(), before)      # set_wrench leaves them
    run(a, pb)
    run(b, pb)
    ma, mb = a.cache_meta(B).cpu().numpy(), b.cache_meta(B).cpu().numpy()
    assert np.array_equal(ma[:, 3], mb[:, 3]) and ma[:, 3].mean() > 0.8   # the same hits as without the wrench


@pytest.mark.parametrize("N", [10, 60, 7])
def test_invalid_wrenches_report_nan_for_their_slot_only(N):
    B = 64
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=30)
    x0, r, mask, xd, mu = [torch.from_numpy(a).to(dev) for a in pb.f32()]
    mask[5] = 0                                       # all-swing problems: one with a bad wrench, one with a good one
    mask[6] = 0
    force, torque = wrenches(B, N, seed=30)
    good = pkg.BatchedMPC(N=N, max_batch=B)
    good.set_wrench(f32(force), f32(torque))
    ref = to_np(*good.solve(x0, r, mask, xd, mu))
    fb, tb = force.copy(), torque.copy()
    bad_slots = [3, 5, 10, 17, 24]
    fb[3, N - 1, 0] = np.nan                          # last stage only
    fb[5, 0, 2] = np.inf                              # all-swing
    tb[10, 0, 1] = -np.inf
    tb[17, N // 2, 2] = np.nan
    fb[24] = np.nan
    bad = pkg.BatchedMPC(N=N, max_batch=B)
    bad.set_wrench(f32(fb), f32(tb))
    out = to_np(*bad.solve(x0, r, mask, xd, mu))
    assert ref["status"][6] == 1 and np.all(np.isfinite(ref["U"]))
    assert np.all(out["status"][bad_slots] == -1)
    rest = np.setdiff1d(np.arange(B), bad_slots)
    assert same(out, ref, rest)


def test_set_wrench_rejects_bad_arguments():
    mpc = pkg.BatchedMPC(N=10, max_batch=8)
    L = _capi.lib()
    t = f32(np.zeros((8, 10, 3)))
    p = C.c_void_p(t.data_ptr())
    for args in ((8, 0, None, p), (8, 0, p, None), (-1, 0, p, p), (8, 1, p, p), (4, -1, p, p)):
        assert L.cmpc_set_wrench(mpc._h, *args, None) == -1        # CMPC_ERR_INVALID
    assert L.cmpc_set_wrench(mpc._h, 0, 0, p, p, None) == 0
    with pytest.raises(ValueError):
        mpc.set_wrench(t[:, :, :2])
    with pytest.raises(ValueError):
        mpc.set_wrench(t, f32(np.zeros((8, 4, 3))))
    mpc.set_wrench(f32(np.ones((8, 1, 3))))                         # broadcast over the stages, zero torque


def test_graph_capture_of_set_wrench():
    B, N = 64, 10
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=31)
    args = [a.to(dev) for a in map(torch.from_numpy, pb.f32())]
    w1, w2 = (tuple(map(f32, wrenches(B, N, seed=s))) for s in (31, 32))
    # the first call allocates: refused inside a capture, which stays valid (here: it captures a plain solve)
    mpc = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0)
    ref = to_np(*run(pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0), pb))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        with pytest.raises(_capi.CmpcError) as ei:
            mpc.set_wrench(*w1)
        U, X, st = mpc.solve(*args)
    assert ei.value.code == -1
    g.replay()
    torch.cuda.synchronize()
    assert same(to_np(U, X, st), ref)
    # after one eager call, set_wrench + solve captured and replayed = eager
    mpc.set_wrench(*w1)
    torch.cuda.synchronize()
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2):
        mpc.set_wrench(*w2)
        U2, X2, st2 = mpc.solve(*args)
    mpc.set_wrench(*w1)
    g2.replay()
    torch.cuda.synchronize()
    eager = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0)
    eager.set_wrench(*w2)
    assert same(to_np(U2, X2, st2), to_np(*run(eager, pb)))


@pytest.mark.parametrize("N,body", [(5, 0), (10, 0), (30, 0), (5, 1), (10, 1), (30, 1)])
def test_condense_with_wrench_matches_oracle(N, body):
    pb = synthetic_batch(6, N=N, gaits=GAIT_NAMES, seed=11)
    force, torque = wrenches(pb.B, N, seed=7)
    m, ib = (r32(a) for a in random_bodies(pb.B, seed=7))
    mpc = pkg.BatchedMPC(N=N, max_batch=pb.B)
    if body:
        mpc.set_body(f32(m), f32(ib))
    mpc.set_wrench(f32(force), f32(torque))
    x0, r, mask, xd, mu = [torch.from_numpy(a).to(dev) for a in pb.f32()]
    H, g = mpc.condense(x0, r, mask, xd)
    torch.cuda.synchronize()
    H, g = H.cpu().numpy().astype(np.float64), g.cpu().numpy().astype(np.float64)
    for b in range(pb.B):
        px0, pr, pst, pxd, _ = pb.problem(b)
        px0, pr, pxd = r32(px0), r32(pr), r32(pxd)
        kw = dict(mass=m[b], ibody_inv=ib[b]) if body else {}
        Ho, go, _, _, idx = wo.condensed_qp(px0, pr, pst, pxd, DT, force[b], torque[b], **kw)
        sel = np.array([12 * i + 3 * l + k for (i, l) in idx for k in range(3)], dtype=int)
        scale = max(np.abs(Ho).max(), 1e-12)
        assert np.abs(H[b][np.ix_(sel, sel)] - Ho).max() <= 2e-5 * scale
        assert np.abs(g[b][sel] - go).max() <= 2e-4 * max(np.abs(go).max(), 1.0)


def test_plant_step_follows_the_predicted_state():
    """One solve with X and one plant step with the same wrench and body: the plant's state is the model's X[:, 1]."""
    B, N = 64, 10
    m, ib = random_bodies(B, seed=9)
    force, torque = random_wrenches(B, N, seed=9)
    ro = pkg.ClosedLoopRollout(B, N=N, gaits=GAIT_NAMES, seed=9, mass=m, ibody_inv=ib, force=force, torque=torque)
    ro.run(25, use_graph=False)                          # a state in motion
    L, h = _capi.lib(), ro.mpc._h
    s = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    P = lambda t: C.c_void_p(t.data_ptr())
    _capi.check(L.cmpc_assemble(h, B, C.byref(ro.gt), P(ro.tick), P(ro.x), P(ro.yaw_start), P(ro.com_start),
                                P(ro.x_des), P(ro.r), P(ro.mask), s))
    U, X, st = ro.mpc.solve(ro.x, ro.r, ro.mask, ro.x_des, ro.mu, want_X=True)
    X1 = X[:, 1].clone()
    assert torch.equal(X[:, 0, :12], ro.x[:, :12])
    _capi.check(L.cmpc_plant_step(h, B, C.byref(ro.gt), P(ro.tick), P(ro.x), P(ro.r), P(U), P(ro.x_des),
                                  P(ro.yaw_start), P(ro.com_start), P(ro.track_err), s))
    torch.cuda.synchronize()
    x, X1 = ro.x.cpu().numpy().astype(np.float64), X1.cpu().numpy().astype(np.float64)
    assert np.all(np.abs(x - X1) <= 2e-5 + 2e-5 * np.abs(X1)), np.abs(x - X1).max()


def test_rollout_balances_a_constant_lateral_push():
    """A constant 15 N lateral push on trotting robots, 1000 ticks: a CUDA graph gives the eager result, and over the
    last two gait cycles the ground forces the controller commands cancel the push on average."""
    B, Fy, T = 256, 15.0, 1000
    force = np.tile([0.0, Fy, 0.0], (B, 1))
    a = pkg.ClosedLoopRollout(B, N=10, gaits=("trot",), seed=7, force=force)
    b = pkg.ClosedLoopRollout(B, N=10, gaits=("trot",), seed=7, force=force)
    cycle = 2 * (10 + 10)                                # trot: two steps of ss + ds ticks
    a.run(T - 2 * cycle, use_graph=True, ticks_per_graph=10)
    b.run(T - 2 * cycle, use_graph=False)
    assert torch.equal(a.x, b.x) and torch.equal(a.out[0], b.out[0])
    fy = torch.zeros(B, dtype=torch.float64, device=dev)
    for _ in range(2 * cycle):
        a.step()
        fy += a.out[0][:, 0, 1::3].sum(1).double()       # stage-0 lateral force of the four legs, what the plant applies
    s = a.summary()
    assert s["finite"] and s["ticks"] == T
    assert 0.15 < s["com_z_min"] and s["com_z_max"] < 0.45
    resid = (fy / (2 * cycle) + Fy).abs().cpu().numpy()
    assert np.all(resid <= 0.05 * Fy), (resid.max(), np.argmax(resid))
