"""Per-robot cost weights (cmpc_set_weights) on the GPU: identity with the configuration's weights, slot weights
against handles configured with the same weights, iterate parity and converged solves against the fp64 oracle given
the same weights, condense, factorisation cache, host paths, invalid weights, graph capture and the closed loop."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import mpc_b200 as pkg                                                      # noqa: E402
from mpc_b200 import _capi                                                  # noqa: E402
from mpc_b200.problems import (synthetic_batch, random_bodies, random_contacts, random_weights, REF_WEIGHTS,   # noqa: E402
                               DT, GAIT_NAMES)
from oracle import condensed_admm as ca, srbd_qp, tight_ipm as ipm         # noqa: E402
import body_oracle as bo                                                    # noqa: E402

ATOL, RTOL = 1e-2, 1e-3
dev = torch.device("cuda", 0)


def f32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)


def r32(a):
    """what the device holds, in fp64 for the oracle"""
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def weights(B, seed):
    return tuple(r32(a) for a in random_weights(B, seed=seed))


def run(mpc, pb, slot0=0):
    U, X, st = mpc.solve(*[a.to(dev) for a in map(torch.from_numpy, pb.f32())], slot0=slot0)
    torch.cuda.synchronize()
    return U, X, st


def to_np(U, X, st):
    return dict(U=U.cpu().numpy().astype(np.float64), X=X.cpu().numpy().astype(np.float64),
                iters=st.iters.cpu().numpy(), status=st.status.cpu().numpy())


def same(a, b, sel=slice(None)):
    return all(np.array_equal(a[k][sel], b[k][sel]) for k in ("U", "X", "iters", "status"))


def config_weights(mpc, B):
    return (np.tile(np.array(mpc.cfg.w[:], dtype=np.float64), (B, 1)), np.full(B, float(mpc.cfg.r_weight)))


def set_config_weights(mpc, B):
    w, rw = config_weights(mpc, B)
    mpc.set_weights(f32(w), f32(rw))


@pytest.mark.parametrize("N,B,variant,cache,extra", [(10, 2048, 0, 0, 0), (12, 64, 0, 0, 0), (30, 64, 0, 0, 0),
                                                     (60, 16, 0, 0, 0), (7, 64, 0, 0, 0), (16, 64, 5, 0, 0),
                                                     (20, 64, 5, 0, 0), (10, 256, 0, 1, 0), (30, 64, 0, 1, 0),
                                                     (10, 256, 0, 0, 1), (4, 64, 0, 0, 0), (5, 64, 0, 0, 0),
                                                     (40, 16, 0, 0, 0), (4, 64, 0, 0, 1), (5, 64, 0, 0, 1),
                                                     (40, 16, 0, 0, 1), (7, 64, 0, 0, 1), (12, 64, 0, 0, 1),
                                                     (16, 64, 5, 0, 1), (20, 64, 5, 0, 1), (30, 64, 0, 1, 1),
                                                     (60, 16, 0, 0, 1)])
def test_configuration_weights_are_bit_identical_to_no_weights(N, B, variant, cache, extra):
    """The WEIGHTS kernels given the configuration's weights reproduce the kernels without weights bit for bit: the
    store kernel builds the handle's M and M^-1 exactly.  At N = 10 with 2048 problems the hardest-first order and
    the reserved-SM launch are active; `extra` gives both handles random bodies and contacts (the
    BODY + CONTACT + WEIGHTS twins against the BODY + CONTACT ones)."""
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=17)
    opts = dict(kernel_variant=variant, cache_factorization=cache, warm_mode=0)
    a = pkg.BatchedMPC(N=N, max_batch=B, **opts)
    b = pkg.BatchedMPC(N=N, max_batch=B, **opts)
    if extra:
        m, ib = random_bodies(B, seed=5)
        c = [f32(x) for x in random_contacts(B, N, seed=5)]
        for h in (a, b):
            h.set_body(f32(m), f32(ib))
            h.set_contact(*c)
    set_config_weights(b, B)
    for _ in range(2 if cache else 1):                # with the cache: the fresh factorisation, then the reuse
        Ua, Xa, sa = run(a, pb)
        Ub, Xb, sb = run(b, pb)
        assert torch.equal(Ua, Ub) and torch.equal(Xa, Xb)
        assert torch.equal(sa.iters, sb.iters) and torch.equal(sa.status, sb.status)
    if cache:
        assert torch.equal(a.cache_meta(B), b.cache_meta(B))


WEIGHT_SETS = [
    (REF_WEIGHTS, 0.0),
    (np.array([2e4, 1e4, 3e4, 1e5, 4e5, 2e5, 5e3, 5e3, 2e4, 3e4, 8e3, 2e4, 5.0]), 1e-4),
    (np.array([5e3, 6e4, 5e3, 6e5, 1e5, 5e5, 3e4, 3e4, 6e3, 1e4, 4e4, 1e4, 0.0]), 1e-2),
    (np.array([1e3, 1e3, 1e3, 1e4, 1e4, 1e4, 1e3, 1e3, 1e3, 1e3, 1e3, 1e3, 1.0]), 1e-3),
]


@pytest.mark.parametrize("N,B", [(10, 2048), (30, 256), (7, 256), (60, 64)])
def test_slot_weights_equal_configured_weights(N, B):
    """A mixed-gait batch at slot0 = 300 with four weight sets assigned to its slots: every problem is bit-identical
    to the same problem on a handle configured with its set (cfg.w, cfg.r_weight)."""
    s0 = 300
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=23)
    k = np.arange(B) % 4
    w = np.stack([WEIGHT_SETS[i][0] for i in k])
    rw = np.array([WEIGHT_SETS[i][1] for i in k])
    mpc = pkg.BatchedMPC(N=N, max_batch=s0 + B, warm_mode=0)
    mpc.set_weights(f32(w), f32(rw), slot0=s0)
    out = to_np(*run(mpc, pb, slot0=s0))
    assert np.mean(out["status"] == 1) >= 0.8
    for i, (wi, rwi) in enumerate(WEIGHT_SETS):
        ref = to_np(*run(pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0, w=wi, r_weight=rwi), pb))
        assert same(out, ref, k == i), i


@pytest.mark.parametrize("N,variant", [(5, 0), (8, 0), (10, 0), (12, 0), (16, 0), (20, 0), (30, 0), (40, 0), (60, 0),
                                       (7, 0), (25, 0), (10, 5), (20, 5), (30, 5)])
def test_iterate_parity_with_random_weights(N, variant):
    B, K = 6, (50 if N < 60 else 120)
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=3)
    w, rw = weights(B, seed=N)
    mpc = pkg.BatchedMPC(N=N, max_batch=B, max_iter=K, check_every=100000, eps_abs=0.0, eps_rel=0.0, warm_mode=0,
                         adaptive_rho_interval=0, kernel_variant=variant)
    mpc.set_weights(f32(w), f32(rw))
    out = to_np(*run(mpc, pb))
    assert np.all(out["iters"] == K)
    for b in range(B):
        x0, r, stance, xd, mu = pb.problem(b)
        H, g, Sc, c0, idx = bo.condensed_qp(x0, r, stance, xd, DT, w=w[b], r_weight=rw[b])
        ref = bo._finish(ca.admm(H, g, mu, fixed_iters=K, rho=float(mpc.cfg.rho), sigma=float(mpc.cfg.sigma),
                                 alpha=float(mpc.cfg.alpha)), r, xd, Sc, c0, idx, H, g)
        err = np.abs(out["U"][b] - ref["U"])
        tr = (3e-3 if N < 60 else 6e-3) * np.abs(ref["U"]).max()
        assert np.all(err <= 2 * ATOL + tr + RTOL * np.abs(ref["U"])), (b, err.max())
        assert np.all(np.abs(out["X"][b].T - ref["X"]) <= 2e-4 + 1e-3 * np.abs(ref["X"]))
        sw = np.repeat(pb.stance[b].reshape(-1) == 0, 3)
        assert np.all(out["U"][b].reshape(-1)[sw] == 0.0)


def weighted_objective(X, U, xd, w, rw):
    return srbd_qp.objective(X, xd, w=w) + rw * float(np.sum(U ** 2))


@pytest.mark.parametrize("N", [10, 30])
def test_converged_solves_with_random_weights(N):
    B = 24
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=12)
    w, rw = weights(B, seed=100 + N)
    mpc = pkg.BatchedMPC(N=N, max_batch=B)
    mpc.set_weights(f32(w), f32(rw))
    out = to_np(*run(mpc, pb))
    assert np.mean(out["status"] == 1) >= 0.9
    for b in range(0, B, 3):
        if out["status"][b] != 1:
            continue
        x0, r, stance, xd, mu = pb.problem(b)
        H, g, Sc, c0, idx = bo.condensed_qp(x0, r, stance, xd, DT, w=w[b], r_weight=rw[b])
        tight = bo._finish(ipm.solve_qp(H, g, mu), r, xd, Sc, c0, idx, H, g)
        J = weighted_objective(out["X"][b].T, out["U"][b], xd, w[b], rw[b])
        Jt = weighted_objective(tight["X"], tight["U"], xd, w[b], rw[b])
        assert abs(J / Jt - 1.0) < 2e-2, (b, J, Jt)


@pytest.mark.parametrize("N,body", [(5, 0), (10, 0), (30, 0), (10, 1)])
def test_condense_with_weights_matches_oracle(N, body):
    pb = synthetic_batch(6, N=N, gaits=GAIT_NAMES, seed=11)
    w, rw = weights(pb.B, seed=7)
    m, ib = (r32(a) for a in random_bodies(pb.B, seed=7))
    mpc = pkg.BatchedMPC(N=N, max_batch=pb.B)
    if body:
        mpc.set_body(f32(m), f32(ib))
    mpc.set_weights(f32(w), f32(rw))
    x0, r, mask, xd, mu = [torch.from_numpy(a).to(dev) for a in pb.f32()]
    H, g = mpc.condense(x0, r, mask, xd)
    torch.cuda.synchronize()
    H, g = H.cpu().numpy().astype(np.float64), g.cpu().numpy().astype(np.float64)
    for b in range(pb.B):
        px0, pr, pst, pxd, _ = pb.problem(b)
        px0, pr, pxd = r32(px0), r32(pr), r32(pxd)
        kw = dict(mass=m[b], ibody_inv=ib[b]) if body else {}
        Ho, go, _, _, idx = bo.condensed_qp(px0, pr, pst, pxd, DT, w=w[b], r_weight=rw[b], **kw)
        sel = np.array([12 * i + 3 * l + k for (i, l) in idx for k in range(3)], dtype=int)
        scale = max(np.abs(Ho).max(), 1e-12)
        assert np.abs(H[b][np.ix_(sel, sel)] - Ho).max() <= 2e-5 * scale
        assert np.abs(g[b][sel] - go).max() <= 2e-4 * max(np.abs(go).max(), 1.0)


def test_set_weights_invalidates_the_factorisation_cache():
    B = 256
    pb = synthetic_batch(B, N=10, gaits=GAIT_NAMES, seed=21)
    w, rw = weights(B, seed=21)
    mpc = pkg.BatchedMPC(N=10, max_batch=B, warm_mode=0, cache_factorization=1, cache_max_iter=1000)
    run(mpc, pb)
    run(mpc, pb)
    assert mpc.cache_meta(B).cpu().numpy()[:, 2].mean() > 0.8          # entries are valid
    mpc.set_weights(f32(w), f32(rw))
    assert np.all(mpc.cache_meta(B).cpu().numpy()[:, 2] == 0)          # set_weights dropped them
    U1, X1, s1 = run(mpc, pb)
    m1 = mpc.cache_meta(B).cpu().numpy()
    assert np.all(m1[:, 3] == 0)                                       # refactorised
    ref = pkg.BatchedMPC(N=10, max_batch=B, warm_mode=0)
    ref.set_weights(f32(w), f32(rw))
    U0, X0, s0 = run(ref, pb)
    assert torch.equal(U1, U0) and torch.equal(s1.iters, s0.iters)     # a miss is the plain path
    U2, X2, s2 = run(mpc, pb)
    m2 = mpc.cache_meta(B).cpu().numpy()
    ok = s1.status.cpu().numpy() == 1
    adapted = m1[:, 0] != np.float32(mpc.cfg.rho)
    assert np.all(m2[ok & ~adapted, 3] == 1)                           # ... and the next solve reuses
    assert torch.equal(U2, U1) and torch.equal(s2.iters, s1.iters)


def test_host_paths_use_the_slot_weights():
    B, N = 2048, 10
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=8)
    w, rw = weights(B, seed=8)

    def handle(**kw):
        h = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0, **kw)
        h.set_weights(f32(w), f32(rw))
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


@pytest.mark.parametrize("N", [10, 60])
def test_invalid_weights_report_nan_for_their_slot_only(N):
    B = 64
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=30)
    w, rw = weights(B, seed=30)
    good = pkg.BatchedMPC(N=N, max_batch=B)
    good.set_weights(f32(w), f32(rw))
    ref = to_np(*run(good, pb))
    wb, rwb = w.copy(), rw.copy()
    bad_slots = [3, 10, 17, 24, 31, 38, 45]
    wb[3, 2] = np.nan                  # non-finite
    wb[10, 4] = -1.0                   # negative
    wb[17, 12] = np.inf                # non-finite, in the unused gravity entry too
    wb[24, 7] = 2.0 * wb[24, 6]        # w[6] != w[7]
    wb[31, 1] = wb[31, 7] = wb[31, 6] = 0.0   # axis 1: position and velocity weight zero
    rwb[38] = np.nan
    rwb[45] = -1e-3
    bad = pkg.BatchedMPC(N=N, max_batch=B)
    bad.set_weights(f32(wb), f32(rwb))
    out = to_np(*run(bad, pb))
    assert np.all(out["status"][bad_slots] == -1)
    rest = np.setdiff1d(np.arange(B), bad_slots)
    assert same(out, ref, rest)


def test_set_weights_rejects_bad_arguments():
    mpc = pkg.BatchedMPC(N=10, max_batch=8)
    L = _capi.lib()
    t = f32(np.tile(REF_WEIGHTS, (8, 1)))
    r = f32(np.zeros(8))
    p, q = C.c_void_p(t.data_ptr()), C.c_void_p(r.data_ptr())
    for args in ((8, 0, None, q), (8, 0, p, None), (-1, 0, p, q), (8, 1, p, q), (4, -1, p, q)):
        assert L.cmpc_set_weights(mpc._h, *args, None) == -1        # CMPC_ERR_INVALID
    assert L.cmpc_set_weights(mpc._h, 0, 0, p, q, None) == 0
    with pytest.raises(ValueError):
        mpc.set_weights(t[:, :12])
    with pytest.raises(ValueError):
        mpc.set_weights(t, f32(np.zeros(3)))


def test_graph_capture_of_set_weights():
    B, N = 64, 10
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=31)
    args = [a.to(dev) for a in map(torch.from_numpy, pb.f32())]
    w1, w2 = (tuple(map(f32, weights(B, seed=s))) for s in (31, 32))
    # the first call allocates: refused inside a capture, which stays valid (here: it captures a plain solve)
    mpc = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0)
    ref = to_np(*run(pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0), pb))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        with pytest.raises(_capi.CmpcError) as ei:
            mpc.set_weights(*w1)
        U, X, st = mpc.solve(*args)
    assert ei.value.code == -1
    g.replay()
    torch.cuda.synchronize()
    assert same(to_np(U, X, st), ref)
    # after one eager call, set_weights + solve captured and replayed = eager
    mpc.set_weights(*w1)
    torch.cuda.synchronize()
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2):
        mpc.set_weights(*w2)
        U2, X2, st2 = mpc.solve(*args)
    mpc.set_weights(*w1)
    g2.replay()
    torch.cuda.synchronize()
    eager = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0)
    eager.set_weights(*w2)
    assert same(to_np(U2, X2, st2), to_np(*run(eager, pb)))


def test_rollout_with_random_weights_graph_equals_eager():
    w, rw = random_weights(256, seed=7)
    a = pkg.ClosedLoopRollout(256, N=10, gaits=GAIT_NAMES, seed=7, w=w, r_weight=rw)
    b = pkg.ClosedLoopRollout(256, N=10, gaits=GAIT_NAMES, seed=7, w=w, r_weight=rw)
    a.run(61, use_graph=True, ticks_per_graph=10)
    b.run(61, use_graph=False)
    sa = a.summary()
    assert torch.equal(a.x, b.x) and torch.equal(a.out[0], b.out[0])
    assert sa["finite"]
    assert 0.15 < sa["com_z_min"] and sa["com_z_max"] < 0.45
