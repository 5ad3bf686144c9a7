"""Per-foot contact surfaces (cmpc_set_contact) on the GPU: identity of flat contacts with no contacts, unset slots,
iterate parity and converged solves against the fp64 contact oracle, per-leg bounds, slot bookkeeping, host paths,
factorisation cache, graph capture and invalid contacts."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import mpc_b200 as pkg                                                      # noqa: E402
from mpc_b200 import _capi                                                  # noqa: E402
from mpc_b200.problems import synthetic_batch, random_bodies, random_contacts, DT, GAIT_NAMES   # noqa: E402
from oracle import srbd_qp                                                  # noqa: E402
import contact_oracle as co                                                 # noqa: E402

ATOL, RTOL = 1e-2, 1e-3
dev = torch.device("cuda", 0)


def f32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)


def r32(a):
    """what the device holds, in fp64 for the oracle"""
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def contacts(B, N, seed):
    return tuple(r32(a) for a in random_contacts(B, N, seed=seed))


def run(mpc, pb, slot0=0):
    U, X, st = mpc.solve(*[a.to(dev) for a in map(torch.from_numpy, pb.f32())], slot0=slot0)
    torch.cuda.synchronize()
    return U, X, st


def to_np(U, X, st):
    return dict(U=U.cpu().numpy().astype(np.float64), X=X.cpu().numpy().astype(np.float64),
                iters=st.iters.cpu().numpy(), status=st.status.cpu().numpy())


def set_flat(mpc, pb, c=1.0, slot0=0):
    """flat ground with the problems' mu and the configuration's bounds"""
    B = pb.B
    mpc.set_contact(f32(np.tile([0.0, 0.0, c], (B, 1, 1, 1))), f32(pb.mu.reshape(B, 1, 1)), slot0=slot0)


def local_forces(U, normal):
    """R' f per leg-stage, (B,N,4,3)"""
    B, N = U.shape[:2]
    return np.einsum("bjlki,bjlk->bjli", co.contact_frame(normal), U.reshape(B, N, 4, 3))


def same(a, b):
    return all(np.array_equal(a[k], b[k]) for k in ("U", "X", "iters", "status"))


@pytest.mark.parametrize("N,B,variant,cache", [(10, 2048, 0, 0), (12, 64, 0, 0), (30, 64, 0, 0), (60, 16, 0, 0),
                                               (7, 64, 0, 0), (16, 64, 5, 0), (20, 64, 5, 0), (10, 256, 0, 1),
                                               (30, 64, 0, 1), (4, 64, 0, 0), (5, 64, 0, 0), (40, 16, 0, 0)])
def test_flat_contacts_are_bit_identical_to_no_contacts(N, B, variant, cache):
    """The CONTACT kernels given flat ground (normal (0,0,1) or (0,0,2.5)), the call's mu and the configuration's
    bounds reproduce the plain kernels bit for bit; at N = 10 with 2048 problems the hardest-first order and the
    reserved-SM launch are active; with the cache over the fresh factorisation and its reuse."""
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=17)
    opts = dict(kernel_variant=variant, cache_factorization=cache, warm_mode=0)
    a = pkg.BatchedMPC(N=N, max_batch=B, **opts)
    handles = []
    for c in (1.0, 2.5):
        h = pkg.BatchedMPC(N=N, max_batch=B, **opts)
        set_flat(h, pb, c)
        handles.append(h)
    for _ in range(2 if cache else 1):
        Ua, Xa, sa = run(a, pb)
        for h in handles:
            Ub, Xb, sb = run(h, pb)
            assert torch.equal(Ua, Ub) and torch.equal(Xa, Xb)
            assert torch.equal(sa.iters, sb.iters) and torch.equal(sa.status, sb.status)
    if cache:
        for h in handles:
            assert torch.equal(a.cache_meta(B), h.cache_meta(B))


@pytest.mark.parametrize("N", [10, 30])
def test_unset_slots_are_unaffected(N):
    B = 2048
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=19)
    ref = to_np(*run(pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0), pb))
    mpc = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0)
    normal, mu, lo, hi = contacts(B // 2, N, seed=19)
    mpc.set_contact(f32(normal), f32(mu), f32(lo), f32(hi), slot0=B // 2)
    out = to_np(*run(mpc, pb))
    half = slice(0, B // 2)
    assert all(np.array_equal(out[k][half], ref[k][half]) for k in ("U", "X", "iters", "status"))
    assert not np.array_equal(out["U"][B // 2:], ref["U"][B // 2:])


@pytest.mark.parametrize("N,variant,body", [(5, 0, 0), (8, 0, 0), (10, 0, 0), (12, 0, 0), (16, 0, 0), (20, 0, 0),
                                            (30, 0, 0), (40, 0, 0), (60, 0, 0), (7, 0, 0), (25, 0, 0), (10, 5, 0),
                                            (20, 5, 0), (30, 5, 0), (10, 0, 1)])
def test_iterate_parity_with_random_contacts(N, variant, body):
    B, K = 6, (50 if N < 60 else 120)
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=3)
    normal, mu, lo, hi = contacts(B, N, seed=N)
    mpc = pkg.BatchedMPC(N=N, max_batch=B, max_iter=K, check_every=100000, eps_abs=0.0, eps_rel=0.0, warm_mode=0,
                         adaptive_rho_interval=0, kernel_variant=variant)
    mpc.set_contact(f32(normal), f32(mu), f32(lo), f32(hi))
    kw = [{} for _ in range(B)]
    if body:
        m, ib = (r32(a) for a in random_bodies(B, seed=N))
        mpc.set_body(f32(m), f32(ib))
        kw = [dict(mass=m[b], ibody_inv=ib[b]) for b in range(B)]
    out = to_np(*run(mpc, pb))
    assert np.all(out["iters"] == K)
    for b in range(B):
        x0, r, stance, xd, _ = pb.problem(b)
        ref = co.admm_solve(x0, r, stance, xd, DT, normal[b], mu[b], lo[b], hi[b], fixed_iters=K,
                            rho=float(mpc.cfg.rho), sigma=float(mpc.cfg.sigma), alpha=float(mpc.cfg.alpha), **kw[b])
        err = np.abs(out["U"][b] - ref["U"])
        tr = (3e-3 if N < 60 else 6e-3) * np.abs(ref["U"]).max()
        assert np.all(err <= 2 * ATOL + tr + RTOL * np.abs(ref["U"])), (b, err.max())
        assert np.all(np.abs(out["X"][b].T - ref["X"]) <= 2e-4 + 1e-3 * np.abs(ref["X"]))
        sw = np.repeat(pb.stance[b].reshape(-1) == 0, 3)
        assert np.all(out["U"][b].reshape(-1)[sw] == 0.0)


def check_feasible(mpc, U, stance, normal, mu, lo, hi):
    """every stance force in its own rotated frustum within 2 (eps_abs + eps_rel max|U|), swing forces exactly 0"""
    loc = local_forces(U, normal)
    on = stance.astype(bool)
    tol = 2.0 * (mpc.cfg.eps_abs + mpc.cfg.eps_rel * np.abs(U).max())
    fn = loc[..., 2][on]
    assert np.all(fn >= lo[on] - tol) and np.all(fn <= hi[on] + tol)
    assert np.all(np.abs(loc[..., :2][on]) <= mu[on][:, None] * fn[:, None] + tol)
    assert np.all(U.reshape(loc.shape)[~on] == 0.0)


@pytest.mark.parametrize("N", [10, 30])
def test_converged_solves_with_random_contacts(N):
    B = 24
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=12)
    normal, mu, lo, hi = contacts(B, N, seed=100 + N)
    mpc = pkg.BatchedMPC(N=N, max_batch=B)
    mpc.set_contact(f32(normal), f32(mu), f32(lo), f32(hi))
    out = to_np(*run(mpc, pb))
    assert np.mean(out["status"] == 1) >= 0.9
    ok = out["status"] == 1
    check_feasible(mpc, out["U"][ok], pb.stance[ok], normal[ok], mu[ok], lo[ok], hi[ok])
    for b in range(0, B, 6):
        if not ok[b]:
            continue
        x0, r, stance, xd, _ = pb.problem(b)
        tight = co.ipm_solve(x0, r, stance, xd, DT, normal[b], mu[b], lo[b], hi[b])
        assert abs(srbd_qp.objective(out["X"][b].T, xd) / tight["J"] - 1.0) < 2e-2, b


def test_each_bound_acts_on_its_own_leg_stage():
    """mu = 0 on one stance leg-stage and f_max = 10 N on another, per problem: the first carries no tangential
    force in its frame, the second at most 10 N along its normal; every other leg-stage keeps its own frustum."""
    B, N = 32, 10
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=23)
    normal, mu, lo, hi = contacts(B, N, seed=23)
    zero_mu, low_max = [], []
    for b in range(B):
        on = np.argwhere(pb.stance[b])
        j0, l0 = on[0]
        j1, l1 = on[len(on) // 2]
        mu[b, j0, l0] = 0.0
        hi[b, j1, l1] = 10.0
        zero_mu.append((b, j0, l0))
        low_max.append((b, j1, l1))
    mpc = pkg.BatchedMPC(N=N, max_batch=B)
    mpc.set_contact(f32(normal), f32(mu), f32(lo), f32(hi))
    out = to_np(*run(mpc, pb))
    ok = out["status"] == 1
    assert ok.mean() >= 0.9
    loc = local_forces(out["U"], normal)
    tol = 2.0 * (mpc.cfg.eps_abs + mpc.cfg.eps_rel * np.abs(out["U"]).max())
    for b, j, l in zero_mu:
        if ok[b]:
            assert np.all(np.abs(loc[b, j, l, :2]) <= tol), (b, loc[b, j, l])
    for b, j, l in low_max:
        if ok[b]:
            assert loc[b, j, l, 2] <= 10.0 + tol, (b, loc[b, j, l])
    assert max(loc[b, j, l, 2] for b, j, l in low_max if ok[b]) > 9.0          # the bound is active somewhere
    check_feasible(mpc, out["U"][ok], pb.stance[ok], normal[ok], mu[ok], lo[ok], hi[ok])


def test_problems_use_the_contact_of_their_slot():
    B, N, s0 = 64, 10, 100
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=27)
    ca_ = contacts(B, N, seed=27)
    cb_ = contacts(B, N, seed=28)
    mpc = pkg.BatchedMPC(N=N, max_batch=s0 + B, warm_mode=0)
    mpc.set_contact(*map(f32, ca_))
    mpc.set_contact(*map(f32, cb_), slot0=s0)
    at0 = to_np(*run(mpc, pb))
    at_s0 = to_np(*run(mpc, pb, slot0=s0))
    for c, got in ((ca_, at0), (cb_, at_s0)):
        ref = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0)
        ref.set_contact(*map(f32, c))
        assert same(got, to_np(*run(ref, pb)))
    assert not np.array_equal(at0["U"], at_s0["U"])


def test_host_paths_use_the_slot_contacts():
    B, N = 2048, 10
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=8)
    c = contacts(B, N, seed=8)

    def handle(**kw):
        h = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0, **kw)
        h.set_contact(*map(f32, c))
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
    check(*handle().solve_host(*hin, out=pinned_out()))                          # zero-copy
    check(*handle(host_zero_copy=0).solve_host(*hin, out=pinned_out()))          # two chunks, engine copies
    check(*handle().solve_host(*pb.f32()))                                       # pageable, staged
    h = handle()
    out = pinned_out()
    h.host_wait(h.solve_host_async(*hin, out=out))
    U, X, it, _, _, stt = out
    check(U, X, type("S", (), dict(iters=it, status=stt)))


def test_set_contact_keeps_the_factorisation_cache():
    B, N = 256, 10
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=21)
    normal, mu, lo, hi = contacts(B, N, seed=21)
    mpc = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0, cache_factorization=1, cache_max_iter=1000)
    _, _, s1 = run(mpc, pb)
    run(mpc, pb)
    m1 = mpc.cache_meta(B).cpu().numpy()
    ok = s1.status.cpu().numpy() == 1
    hits = ok & (m1[:, 0] == np.float32(mpc.cfg.rho)) & (m1[:, 3] == 1)
    assert hits.mean() > 0.5
    mpc.set_contact(f32(normal), f32(mu), f32(lo), f32(hi))
    assert np.array_equal(mpc.cache_meta(B).cpu().numpy()[:, 2], m1[:, 2])      # entries stay valid
    out = to_np(*run(mpc, pb))
    m2 = mpc.cache_meta(B).cpu().numpy()
    assert np.all(m2[hits, 3] == 1)                                            # ... and are reused
    assert np.mean(out["status"] == 1) >= 0.9
    for b in np.flatnonzero(hits & (out["status"] == 1))[:4]:
        x0, r, stance, xd, _ = pb.problem(b)
        tight = co.ipm_solve(x0, r, stance, xd, DT, normal[b], mu[b], lo[b], hi[b])
        assert abs(srbd_qp.objective(out["X"][b].T, xd) / tight["J"] - 1.0) < 2e-2, b


def test_graph_capture_of_set_contact():
    B, N = 64, 10
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=31)
    args = [a.to(dev) for a in map(torch.from_numpy, pb.f32())]
    c1, c2 = (tuple(map(f32, contacts(B, N, seed=s))) for s in (31, 32))
    # the first call allocates: refused inside a capture, which stays valid (here: it captures a plain solve)
    mpc = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0)
    ref = to_np(*run(pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0), pb))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        with pytest.raises(_capi.CmpcError) as ei:
            mpc.set_contact(*c1)
        U, X, st = mpc.solve(*args)
    assert ei.value.code == -1
    g.replay()
    torch.cuda.synchronize()
    assert same(to_np(U, X, st), ref)
    # after one eager call, set_contact + solve captured and replayed = eager
    mpc.set_contact(*c1)
    torch.cuda.synchronize()
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2):
        mpc.set_contact(*c2)
        U2, X2, st2 = mpc.solve(*args)
    mpc.set_contact(*c1)
    g2.replay()
    torch.cuda.synchronize()
    eager = pkg.BatchedMPC(N=N, max_batch=B, warm_mode=0)
    eager.set_contact(*c2)
    assert same(to_np(U2, X2, st2), to_np(*run(eager, pb)))


def test_invalid_contacts_report_nan_for_their_slot_only():
    B, N = 64, 10
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=30)
    normal, mu, lo, hi = contacts(B, N, seed=30)
    good = pkg.BatchedMPC(N=N, max_batch=B)
    good.set_contact(f32(normal), f32(mu), f32(lo), f32(hi))
    ref = to_np(*run(good, pb))
    nb, mb, lb, hb = normal.copy(), mu.copy(), lo.copy(), hi.copy()
    swing = tuple(np.argwhere(pb.stance[3] == 0)[0])       # an invalid swing leg-stage fails its slot too
    nb[(3,) + swing] = np.nan
    nb[5, 2, 1] = [0.0, 0.0, 5e-7]
    mb[7, 0, 0] = -0.1
    mb[9, 4, 3] = np.inf
    lb[11, 1, 2] = -1.0
    lb[13, 3, 0] = hb[13, 3, 0] + 1.0
    hb[15, 9, 1] = np.inf
    bad_slots = [3, 5, 7, 9, 11, 13, 15]
    bad = pkg.BatchedMPC(N=N, max_batch=B)
    bad.set_contact(f32(nb), f32(mb), f32(lb), f32(hb))
    out = to_np(*run(bad, pb))
    assert np.all(out["status"][bad_slots] == -1)
    rest = np.setdiff1d(np.arange(B), bad_slots)
    for k in ("U", "X", "iters", "status"):
        assert np.array_equal(out[k][rest], ref[k][rest]), k
