"""Per-robot mass and body inertia (cmpc_set_body) on the GPU: identity with the configuration's body,
iterate parity and converged solves against the fp64 oracle given the same bodies, slot bookkeeping,
condense / plant / closed loop / host paths, factorisation cache and invalid bodies."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import mpc_b200 as pkg                                                      # noqa: E402
from mpc_b200 import _capi                                                  # noqa: E402
from mpc_b200.problems import (synthetic_batch, random_bodies, DT, GAIT_NAMES, GRAVITY,   # noqa: E402
                               NOMINAL_COM, NOMINAL_FEET)
from mpc_b200.solver import _ptr                                            # noqa: E402
from oracle import condensed_admm as ca, srbd_qp                            # noqa: E402
import body_oracle as bo                                                    # noqa: E402

ATOL, RTOL = 1e-2, 1e-3
dev = torch.device("cuda", 0)


def close(a, b, atol=ATOL, rtol=RTOL):
    return np.all(np.abs(a - b) <= atol + rtol * np.abs(b))


def f32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)


def bodies(B, seed):
    """random_bodies rounded to fp32 (what the device holds), in fp64 for the oracle."""
    m, ib = random_bodies(B, seed=seed)
    return m.astype(np.float32).astype(np.float64), ib.astype(np.float32).astype(np.float64)


def config_body(mpc, B):
    return (np.full(B, mpc.cfg.mass, dtype=np.float64),
            np.tile(np.diag(np.array(mpc.cfg.ibody_inv[:], dtype=np.float64)), (B, 1, 1)))


def run(mpc, pb, slot0=0):
    U, X, st = mpc.solve(*[a.to(dev) for a in map(torch.from_numpy, pb.f32())], slot0=slot0)
    torch.cuda.synchronize()
    return U, X, st


def to_np(U, X, st):
    return dict(U=U.cpu().numpy().astype(np.float64), X=X.cpu().numpy().astype(np.float64),
                iters=st.iters.cpu().numpy(), status=st.status.cpu().numpy())


@pytest.mark.parametrize("N,B,variant,cache", [(10, 2048, 0, 0), (12, 64, 0, 0), (30, 64, 0, 0), (60, 16, 0, 0),
                                               (7, 64, 0, 0), (16, 64, 5, 0), (20, 64, 5, 0), (10, 256, 0, 1),
                                               (30, 64, 0, 1), (4, 64, 0, 0), (5, 64, 0, 0), (40, 16, 0, 0)])
def test_configuration_body_is_bit_identical_to_no_body(N, B, variant, cache):
    """The BODY kernels given the configuration's body reproduce the plain kernels bit for bit (the full-matrix
    leg map adds exact zeros for a diagonal inertia); at N = 10 with 2048 problems the hardest-first order and
    the reserved-SM launch are active."""
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=17)
    opts = dict(kernel_variant=variant, cache_factorization=cache, warm_mode=0)
    a = pkg.BatchedMPC(N=N, max_batch=B, **opts)
    b = pkg.BatchedMPC(N=N, max_batch=B, **opts)
    m, ib = config_body(b, B)
    b.set_body(f32(m), f32(ib))
    for _ in range(2 if cache else 1):                # with the cache: the fresh factorisation, then the reuse
        Ua, Xa, sa = run(a, pb)
        Ub, Xb, sb = run(b, pb)
        assert torch.equal(Ua, Ub) and torch.equal(Xa, Xb)
        assert torch.equal(sa.iters, sb.iters) and torch.equal(sa.status, sb.status)
    if cache:
        assert torch.equal(a.cache_meta(B), b.cache_meta(B))


@pytest.mark.parametrize("N,variant", [(5, 0), (8, 0), (10, 0), (12, 0), (16, 0), (20, 0), (30, 0), (40, 0), (60, 0),
                                       (7, 0), (25, 0), (10, 5), (20, 5), (30, 5)])
def test_iterate_parity_with_random_bodies(N, variant):
    B, K = 6, (50 if N < 60 else 120)
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=3)
    m, ib = bodies(B, seed=N)
    mpc = pkg.BatchedMPC(N=N, max_batch=B, max_iter=K, check_every=100000, eps_abs=0.0, eps_rel=0.0, warm_mode=0,
                         adaptive_rho_interval=0, kernel_variant=variant)
    mpc.set_body(f32(m), f32(ib))
    out = to_np(*run(mpc, pb))
    assert np.all(out["iters"] == K)
    for b in range(B):
        x0, r, stance, xd, mu = pb.problem(b)
        ref = bo.admm_solve(x0, r, stance, xd, mu, DT, m[b], ib[b], fixed_iters=K, rho=float(mpc.cfg.rho),
                            sigma=float(mpc.cfg.sigma), alpha=float(mpc.cfg.alpha))
        err = np.abs(out["U"][b] - ref["U"])
        tr = (3e-3 if N < 60 else 6e-3) * np.abs(ref["U"]).max()
        assert np.all(err <= 2 * ATOL + tr + RTOL * np.abs(ref["U"])), (b, err.max())
        assert close(out["X"][b].T, ref["X"], atol=2e-4, rtol=1e-3)
        sw = np.repeat(pb.stance[b].reshape(-1) == 0, 3)
        assert np.all(out["U"][b].reshape(-1)[sw] == 0.0)


@pytest.mark.parametrize("N", [10, 30])
def test_converged_solves_with_random_bodies(N):
    B = 24
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=12)
    m, ib = bodies(B, seed=100 + N)
    mpc = pkg.BatchedMPC(N=N, max_batch=B)
    mpc.set_body(f32(m), f32(ib))
    out = to_np(*run(mpc, pb))
    assert np.mean(out["status"] == 1) >= 0.9
    for b in range(0, B, 6):
        if out["status"][b] != 1:
            continue
        x0, r, stance, xd, mu = pb.problem(b)
        tight = bo.ipm_solve(x0, r, stance, xd, mu, DT, m[b], ib[b])
        assert abs(srbd_qp.objective(out["X"][b].T, xd) / tight["J"] - 1.0) < 2e-2, b


def test_each_problem_holds_its_own_slots_weight():
    """Identical standing problems (x0 = x_des, four feet down, at rest) at slot0 != 0 with masses of 6-12 kg:
    the zero-cost optimum holds each robot's weight, sum f_z(stage 0) = m g.  With the hardest-first order
    (which depends on the mass through the score) any mix-up of slots and ranks shows."""
    B, N, s0 = 1536, 10, 300
    x0 = np.zeros(13); x0[3:6] = NOMINAL_COM; x0[12] = GRAVITY
    xd = np.tile(x0, (B, N + 1, 1))
    r = np.tile(NOMINAL_FEET - NOMINAL_COM, (B, N, 1, 1))
    args = [f32(np.tile(x0, (B, 1))), f32(r), torch.full((B, N), 15, dtype=torch.uint8, device=dev), f32(xd),
            f32(np.full(B, 0.8))]
    mass = np.random.default_rng(4).permutation(np.linspace(6.0, 12.0, B))
    mpc = pkg.BatchedMPC(N=N, max_batch=s0 + B, eps_abs=1e-5, eps_rel=1e-5, max_iter=4000)
    mpc.set_body(f32(mass), f32(np.tile(np.diag([1 / 0.24, 1.0, 1.0]), (B, 1, 1))), slot0=s0)
    U, _, st = mpc.solve(*args, slot0=s0)
    torch.cuda.synchronize()
    fz = U.cpu().numpy()[:, 0, 2::3].sum(1)
    m32 = mass.astype(np.float32).astype(np.float64)
    assert np.all(np.abs(fz / (m32 * 9.81) - 1.0) < 1e-2), np.abs(fz / (m32 * 9.81) - 1.0).max()


@pytest.mark.parametrize("N", [5, 10, 30])
def test_condense_with_bodies_matches_oracle(N):
    pb = synthetic_batch(6, N=N, gaits=GAIT_NAMES, seed=11)
    m, ib = bodies(pb.B, seed=7)
    mpc = pkg.BatchedMPC(N=N, max_batch=pb.B)
    mpc.set_body(f32(m), f32(ib))
    x0, r, mask, xd, mu = [torch.from_numpy(a).to(dev) for a in pb.f32()]
    H, g = mpc.condense(x0, r, mask, xd)
    torch.cuda.synchronize()
    H, g = H.cpu().numpy().astype(np.float64), g.cpu().numpy().astype(np.float64)
    for b in range(pb.B):
        px0, pr, pst, pxd, _ = pb.problem(b)
        px0, pr, pxd = (np.float32(px0).astype(np.float64), np.float32(pr).astype(np.float64),
                        np.float32(pxd).astype(np.float64))
        Ho, go, _, _, idx = bo.condensed_qp(px0, pr, pst, pxd, DT, mass=m[b], ibody_inv=ib[b])
        sel = np.array([12 * i + 3 * l + k for (i, l) in idx for k in range(3)], dtype=int)
        scale = max(np.abs(Ho).max(), 1e-12)
        assert np.abs(H[b][np.ix_(sel, sel)] - Ho).max() <= 2e-5 * scale
        assert np.abs(g[b][sel] - go).max() <= 2e-4 * max(np.abs(go).max(), 1.0)


def test_set_body_invalidates_the_factorisation_cache():
    B = 256
    pb = synthetic_batch(B, N=10, gaits=GAIT_NAMES, seed=21)
    m, ib = bodies(B, seed=21)
    mpc = pkg.BatchedMPC(N=10, max_batch=B, warm_mode=0, cache_factorization=1, cache_max_iter=1000)
    run(mpc, pb)
    run(mpc, pb)
    assert mpc.cache_meta(B).cpu().numpy()[:, 2].mean() > 0.8          # entries are valid
    mpc.set_body(f32(m), f32(ib))
    assert np.all(mpc.cache_meta(B).cpu().numpy()[:, 2] == 0)          # set_body dropped them
    U1, X1, s1 = run(mpc, pb)
    m1 = mpc.cache_meta(B).cpu().numpy()
    assert np.all(m1[:, 3] == 0)                                       # refactorised
    ref = pkg.BatchedMPC(N=10, max_batch=B, warm_mode=0)
    ref.set_body(f32(m), f32(ib))
    U0, X0, s0 = run(ref, pb)
    assert torch.equal(U1, U0) and torch.equal(s1.iters, s0.iters)     # a miss is the plain path
    U2, X2, s2 = run(mpc, pb)
    m2 = mpc.cache_meta(B).cpu().numpy()
    ok = s1.status.cpu().numpy() == 1
    adapted = m1[:, 0] != np.float32(mpc.cfg.rho)
    assert np.all(m2[ok & ~adapted, 3] == 1)                           # ... and the next solve reuses
    assert torch.equal(U2, U1) and torch.equal(s2.iters, s1.iters)


def test_plant_step_uses_each_robots_body():
    B = 32
    m, ib = bodies(B, seed=2)
    ro = pkg.ClosedLoopRollout(B, N=10, seed=2, mass=m, ibody_inv=ib)
    rng = np.random.default_rng(3)
    x = rng.normal(0, 0.3, (B, 13)); x[:, 12] = GRAVITY
    U = rng.uniform(-20, 60, (B, 10, 12)); r = rng.normal(0, 0.2, (B, 10, 4, 3))
    ro.x.copy_(torch.from_numpy(x.astype(np.float32)))
    ro.r.copy_(torch.from_numpy(r.astype(np.float32)))
    ro.out[0].copy_(torch.from_numpy(U.astype(np.float32)))
    ro.x_des.zero_()
    ro.tick.fill_(40)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _capi.check(_capi.lib().cmpc_plant_step(ro.mpc._h, ro.B, C.byref(ro.gt), _ptr(ro.tick), _ptr(ro.x), _ptr(ro.r),
                                            _ptr(ro.out[0]), _ptr(ro.x_des), _ptr(ro.yaw_start),
                                            _ptr(ro.com_start), _ptr(ro.track_err), s))
    torch.cuda.synchronize()
    xn = ro.x.cpu().numpy()
    xf, rf, Uf = x.astype(np.float32).astype(float), r.astype(np.float32).astype(float), U.astype(np.float32).astype(float)
    for b in range(B):
        Bm = bo.continuous_B(xf[b, 2], rf[b, 0], mass=m[b], ibody_inv=ib[b])
        ref = xf[b] + DT * (srbd_qp.continuous_A(xf[b, 2]) @ xf[b] + Bm @ Uf[b, 0])
        np.testing.assert_allclose(xn[b], ref, atol=2e-5, rtol=1e-5)


def test_closed_loop_with_bodies_matches_fp64_loop():
    from test_gpu_rollout import host_assemble
    B, T = 4, 15
    m, ib = bodies(B, seed=5)
    ro = pkg.ClosedLoopRollout(B, N=10, seed=5, mu=(0.5, 1.0), mass=m, ibody_inv=ib)
    x = ro.x.cpu().numpy().astype(np.float64)
    ys = np.zeros(B); cs = ro.com_start.cpu().numpy().astype(np.float64)
    warm = [None] * B
    for t in range(T):
        xd, r, stance = host_assemble(ro, t, x, ys, cs)
        for b in range(B):
            H, g, Sc, c0, idx = bo.condensed_qp(x[b], r[b], stance[b], xd[b].T, DT, mass=m[b], ibody_inv=ib[b])
            xw = None if warm[b] is None else np.concatenate([warm[b][i, 3 * l:3 * l + 3] for (i, l) in idx])
            res = ca.admm(H, g, ro.mu_host[b], check_every=5, x=xw, rho=0.5, adaptive_interval=25,
                          adaptive_tolerance=3.0, rho_lim=(0.05, 300.0))
            U = np.zeros((10, 12))
            for s_, (i, l) in enumerate(idx):
                U[i, 3 * l:3 * l + 3] = res["x"][3 * s_:3 * s_ + 3]
            warm[b] = U
            Bm = bo.continuous_B(x[b, 2], r[b, 0], mass=m[b], ibody_inv=ib[b])
            x[b] = x[b] + DT * (srbd_qp.continuous_A(x[b, 2]) @ x[b] + Bm @ U[0])
        cs = cs + ro.v_ref.cpu().numpy().astype(np.float64) * DT
        ro.step()
    torch.cuda.synchronize()
    xg = ro.x.cpu().numpy()
    np.testing.assert_allclose(xg[:, 3:6], x[:, 3:6], atol=2e-4)
    np.testing.assert_allclose(xg[:, 9:12], x[:, 9:12], atol=3e-3)
    np.testing.assert_allclose(xg[:, 0:3], x[:, 0:3], atol=2e-3)


def test_rollout_with_random_bodies_graph_equals_eager():
    m, ib = random_bodies(256, seed=7)
    a = pkg.ClosedLoopRollout(256, N=10, gaits=GAIT_NAMES, seed=7, mass=m, ibody_inv=ib)
    b = pkg.ClosedLoopRollout(256, N=10, gaits=GAIT_NAMES, seed=7, mass=m, ibody_inv=ib)
    a.run(61, use_graph=True, ticks_per_graph=10)
    b.run(61, use_graph=False)
    sa = a.summary()
    assert torch.equal(a.x, b.x) and torch.equal(a.out[0], b.out[0])
    assert sa["finite"] and sa["unsolved"] == 0
    assert 0.2 < sa["com_z_min"] and sa["com_z_max"] < 0.4


def test_host_paths_use_the_slot_bodies():
    B, N = 2048, 10
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=8)
    m, ib = bodies(B, seed=8)

    def handle(**kw):
        h = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0, **kw)
        h.set_body(f32(m), f32(ib))
        torch.cuda.synchronize()
        return h
    ref = to_np(*run(handle(), pb))
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    zeros = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory().numpy()

    def pinned_out():
        return (zeros((B, N, 12), torch.float32), zeros((B, N + 1, 13), torch.float32), zeros((B,), torch.int32),
                zeros((B,), torch.float32), zeros((B,), torch.float32), zeros((B,), torch.int32))

    def same(U, X, st):
        assert np.array_equal(U, ref["U"].astype(np.float32)) and np.array_equal(X, ref["X"].astype(np.float32))
        assert np.array_equal(st.iters, ref["iters"]) and np.array_equal(st.status, ref["status"])
    hin = [pin(a) for a in pb.f32()]
    same(*handle().solve_host(*hin, out=pinned_out()))                          # zero-copy
    same(*handle(host_zero_copy=0).solve_host(*hin, out=pinned_out()))          # two chunks, engine copies
    same(*handle().solve_host(*pb.f32()))                                       # pageable, staged
    h = handle()
    out = pinned_out()
    h.host_wait(h.solve_host_async(*hin, out=out))
    U, X, it, _, _, stt = out
    same(U, X, type("S", (), dict(iters=it, status=stt)))


def test_invalid_body_reports_nan_for_its_slot_only():
    B = 64
    pb = synthetic_batch(B, N=10, gaits=GAIT_NAMES, seed=30)
    m, ib = bodies(B, seed=30)
    good = pkg.BatchedMPC(N=10, max_batch=B)
    good.set_body(f32(m), f32(ib))
    ref = to_np(*run(good, pb))
    m_bad, ib_bad = m.copy(), ib.copy()
    m_bad[3] = 0.0
    ib_bad[10, 1, 2] = np.nan
    bad = pkg.BatchedMPC(N=10, max_batch=B)
    bad.set_body(f32(m_bad), f32(ib_bad))
    out = to_np(*run(bad, pb))
    assert out["status"][3] == -1 and out["status"][10] == -1
    rest = np.setdiff1d(np.arange(B), [3, 10])
    for k in ("U", "X", "iters", "status"):
        assert np.array_equal(out[k][rest], ref[k][rest]), k
