"""Every per-slot feature on one handle (cmpc_set_body + cmpc_set_contact + cmpc_set_weights + cmpc_set_wrench): the
BODY + CONTACT + WEIGHTS solve kernels against the composed fp64 oracle (mix_oracle.py) iterate for iterate, their
reserved-SM launch against the plain one, and the termination test of every SOLVED status recomputed in fp64 for
each kind of solve kernel."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import mpc_b200 as pkg                                                      # noqa: E402
from mpc_b200.problems import (synthetic_batch, random_bodies, random_contacts, random_weights,  # noqa: E402
                               random_wrenches, GAIT_NAMES)
import mix_oracle as mo                                                     # noqa: E402

ATOL, RTOL = 1e-2, 1e-3
dev = torch.device("cuda", 0)
r32 = mo.r32
ALL = ("body", "contact", "weights", "wrench")


def f32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)


def draw(B, N, seed, which=ALL):
    """random per-slot features (mix_oracle's `feats`) of the groups in `which`"""
    f = {}
    if "body" in which:
        f.update(zip(("mass", "ibody_inv"), random_bodies(B, seed=seed)))
    if "contact" in which:
        f.update(zip(("normal", "mu", "f_min", "f_max"), random_contacts(B, N, seed=seed)))
    if "weights" in which:
        f.update(zip(("w", "r_weight"), random_weights(B, seed=seed)))
    if "wrench" in which:
        f.update(zip(("force", "torque"), random_wrenches(B, N, seed=seed)))
    return {k: r32(v) for k, v in f.items()}


def put(mpc, f, lo=0, hi=None, slot0=0):
    """give slots [slot0, slot0 + hi - lo) the features of problems [lo, hi)"""
    g = {k: f32(v[lo:hi]) for k, v in f.items()}
    if "mass" in g:
        mpc.set_body(g["mass"], g["ibody_inv"], slot0=slot0)
    if "normal" in g:
        mpc.set_contact(g["normal"], g["mu"], g["f_min"], g["f_max"], slot0=slot0)
    if "w" in g:
        mpc.set_weights(g["w"], g["r_weight"], slot0=slot0)
    if "force" in g:
        mpc.set_wrench(g["force"], g["torque"], slot0=slot0)


def run(mpc, pb, slot0=0):
    U, X, st = mpc.solve(*[a.to(dev) for a in map(torch.from_numpy, pb.f32())], slot0=slot0)
    torch.cuda.synchronize()
    return dict(U=U.cpu().numpy().astype(np.float64), X=X.cpu().numpy().astype(np.float64),
                iters=st.iters.cpu().numpy(), status=st.status.cpu().numpy(),
                pri=st.pri_res.cpu().numpy(), dua=st.dua_res.cpu().numpy())


KEYS = ("U", "X", "iters", "status", "pri", "dua")


# ---- (a) iterate parity of the BODY + CONTACT + WEIGHTS kernels -------------------------------------------------------
@pytest.mark.parametrize("N,variant,which", [(4, 0, ALL), (5, 0, ALL), (8, 0, ALL), (10, 0, ALL), (12, 0, ALL),
                                             (16, 0, ALL), (20, 0, ALL), (30, 0, ALL), (40, 0, ALL), (60, 0, ALL),
                                             (7, 0, ALL), (25, 0, ALL), (10, 5, ALL), (20, 5, ALL), (30, 5, ALL),
                                             (10, 0, ALL[1:]), (30, 0, ALL[1:]), (10, 0, ALL[:3]), (30, 0, ALL[:3])])
def test_iterate_parity_with_all_features(N, variant, which):
    """Random bodies, contacts, weights (r_weight > 0 on odd problems) and wrenches on one handle, K iterations at a
    fixed rho: the same ADMM in fp64 on the same QP.  Without a body the kernels run on the configuration's body that
    the handle gives every slot; without a wrench X is the plain prediction.  Tolerances of the single-feature
    parity tests."""
    B, K = 6, (50 if N < 60 else 120)
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=3)
    f = draw(B, N, seed=N, which=which)
    mpc = pkg.BatchedMPC(N=N, max_batch=B, max_iter=K, check_every=100000, eps_abs=0.0, eps_rel=0.0, warm_mode=0,
                         adaptive_rho_interval=0, kernel_variant=variant)
    put(mpc, f)
    out = run(mpc, pb)
    assert np.all(out["iters"] == K)
    for b in range(B):
        ref = mo.mix_admm(pb, b, f, fixed_iters=K, rho=float(mpc.cfg.rho), sigma=float(mpc.cfg.sigma),
                          alpha=float(mpc.cfg.alpha))
        err = np.abs(out["U"][b] - ref["U"])
        tr = (3e-3 if N < 60 else 6e-3) * np.abs(ref["U"]).max()
        assert np.all(err <= 2 * ATOL + tr + RTOL * np.abs(ref["U"])), (b, err.max())
        assert np.all(np.abs(out["X"][b].T - ref["X"]) <= 2e-4 + 1e-3 * np.abs(ref["X"]))
        sw = np.repeat(pb.stance[b].reshape(-1) == 0, 3)
        assert np.all(out["U"][b].reshape(-1)[sw] == 0.0)


# ---- (b) the reserved-SM launch of the BODY + CONTACT + WEIGHTS kernel ------------------------------------------------
@pytest.mark.timeout(300)
def test_reserved_sm_launch_with_all_features_is_transparent():
    """N = 10 batches of 2048 and 3000 problems with all four features (1.5-4 waves: the hardest-first order, scored
    with the slots' weights, and the reserved-SM rank assignment) equal, bit for bit, the same problems solved in
    slices of 500 at their slots on a second handle with the same per-slot data (plain launches in batch order).  A
    CTA that read its features by launch rank instead of slot would differ."""
    S, N = 3000, 10
    pb = synthetic_batch(S, N=N, gaits=GAIT_NAMES, seed=41)
    f = draw(S, N, seed=41)
    ref = pkg.BatchedMPC(N=N, max_batch=S, warm_mode=0)
    put(ref, f)
    parts = [run(ref, pb.slice(a, min(a + 500, S)), slot0=a) for a in range(0, S, 500)]
    want = {k: np.concatenate([p[k] for p in parts]) for k in KEYS}
    mpc = pkg.BatchedMPC(N=N, max_batch=S, warm_mode=0)
    put(mpc, f)
    for B in (2048, S):
        got = run(mpc, pb.slice(0, B))
        for k in KEYS:
            assert np.array_equal(got[k], want[k][:B], equal_nan=True), (B, k)
    assert np.mean(want["status"] == 1) >= 0.9


# ---- (c) every SOLVED status, recomputed in fp64 ----------------------------------------------------------------------
def check_solved(mpc, pb, f, out, slot0=0):
    """For every problem reported solved, from the returned U (x on the stance legs) and the dual y (get_warm), with
    z = P(x) the projection onto the product of the rotated frustums and H, g of the slot's QP (mix_oracle.mix_qp).

    The kernel stops on |x - z'|_inf <= eps_p with the ADMM's own z' in C, which the library does not return.  P(x) is
    the point of C nearest to x, so per leg |x - P(x)|_2 <= |x - z'|_2 <= sqrt(3) |x - z'|_inf: on a rotated frustum
    |x - P(x)|_inf itself may exceed eps_p (measured on a B200: up to 1.12 eps_p), and the primal checks below are on
    each leg's Euclidean distance to its frustum.

    1. the termination test in fp64: each leg's |x - z|_2 <= sqrt(3) eps_p and |Hx + g + y|_inf <= eps_d with the
       kernel's eps_p = eps_abs + eps_rel max(|x|, |z|), eps_d = eps_abs + eps_rel max(|Hx|, |y|, |g|); 1e-4 relative
       slack for the fp32 evaluation of the same test (as in test_converged_solve_meets_reference_eps);
    2. the reported residuals are those of the returned iterate: dua_res is |Hx + g + y| to 5 % of eps_d (the dual
       residual depends on x and y only), and each leg's |x - z|_2 <= sqrt(3) pri_res + 5 % of eps_p;
    3. y is a multiplier of C: y lies in the normal cone of C at z' (z' = P(z' + y / rho) for the final rho), so by
       the non-expansiveness of P, |P(z + s y) - z| <= 2 |z - z'|_2 <= 2 sqrt(3) pri_res for any s >= 0; checked at
       s = 1 / rho_min with 1e-4 (1 + |z|) for the fp32 rounding of y and z'.  (A bound on y.(x - z) adds nothing to
       this: it sums one term of size |y_l| eps_p per stance leg, so it grows with the horizon.)"""
    B, N = pb.B, pb.N
    yw = mpc.get_warm(B, slot0)[1]
    torch.cuda.synchronize()
    yw = yw.cpu().numpy().astype(np.float64)
    eps_abs, eps_rel, rho_min = float(mpc.cfg.eps_abs), float(mpc.cfg.eps_rel), float(mpc.cfg.rho_min)
    ok = out["status"] == 1
    assert ok.mean() >= 0.9, ok.mean()
    for b in np.flatnonzero(ok):
        H, g, Sc, c0, idx, legs = mo.mix_qp(pb, b, f, as_f32=True)
        if not len(idx):
            continue
        x = np.concatenate([out["U"][b][i, 3 * l:3 * l + 3] for (i, l) in idx])
        y = np.concatenate([yw[b][i, l] for (i, l) in idx])
        z = mo.project(x, legs)
        Hx = H @ x
        pri = np.linalg.norm((x - z).reshape(-1, 3), axis=1).max()          # the largest leg distance to C
        dua = np.abs(Hx + g + y).max()
        eps_p = eps_abs + eps_rel * max(np.abs(x).max(), np.abs(z).max())
        eps_d = eps_abs + eps_rel * max(np.abs(Hx).max(), np.abs(y).max(), np.abs(g).max())
        assert pri <= np.sqrt(3.0) * eps_p * (1 + 1e-4), (b, pri, eps_p)
        assert dua <= eps_d * (1 + 1e-4), (b, dua, eps_d)
        assert abs(out["dua"][b] - dua) <= 0.05 * eps_d, (b, out["dua"][b], dua, eps_d)
        assert pri <= np.sqrt(3.0) * out["pri"][b] + 0.05 * eps_p, (b, pri, out["pri"][b], eps_p)
        moved = np.abs(mo.project(z + y / rho_min, legs) - z).max()
        assert moved <= 2.0 * np.sqrt(3.0) * out["pri"][b] + 1e-4 * (1 + np.abs(z).max()), (b, moved, out["pri"][b])


@pytest.mark.parametrize("N,variant", [(5, 0), (10, 0), (30, 0), (60, 0), (7, 0), (10, 5), (20, 5)])
def test_solved_status_meets_the_termination_test(N, variant):
    """Default settings (eps 1e-3, rho adaptation on, so refactorisations after a rho change run too), 64 mixed-gait
    problems with mu in [0.3, 1] and all four features."""
    B = 64
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=50 + N, mu=(0.3, 1.0))
    f = draw(B, N, seed=50 + N)
    mpc = pkg.BatchedMPC(N=N, max_batch=B, kernel_variant=variant)
    put(mpc, f)
    check_solved(mpc, pb, f, run(mpc, pb))


@pytest.mark.parametrize("N", [10, 30])
def test_solved_status_with_the_factorisation_cache(N):
    """The cached kernels: the fresh factorisation, its reuse by a second solve of the same problems, and its reuse
    after set_contact gives the slots new surfaces (the cached factor does not depend on the contacts).  A re-solve
    of the same problems reuses exactly the entries that are valid and were factorised at the configured rho (rho
    adaptation leaves the factor of its last rho in the cache, which the next solve, starting at the configured rho,
    does not take)."""
    B = 64
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=60 + N, mu=(0.3, 1.0))
    f = draw(B, N, seed=60 + N)
    mpc = pkg.BatchedMPC(N=N, max_batch=B, cache_factorization=1, cache_max_iter=1000)
    put(mpc, f)

    def solve_with_reuse():
        m = mpc.cache_meta(B).cpu().numpy()
        usable = (m[:, 2] == 1) & (m[:, 0] == np.float32(mpc.cfg.rho))
        out = run(mpc, pb)
        reused = mpc.cache_meta(B).cpu().numpy()[:, 3] == 1
        assert usable.any() and np.array_equal(reused, usable), (usable.sum(), reused.sum())
        return out
    check_solved(mpc, pb, f, run(mpc, pb))
    check_solved(mpc, pb, f, solve_with_reuse())
    f2 = dict(f, **draw(B, N, seed=70 + N, which=("contact",)))
    put(mpc, {k: f2[k] for k in ("normal", "mu", "f_min", "f_max")})
    check_solved(mpc, pb, f2, solve_with_reuse())


@pytest.mark.timeout(300)
def test_solved_status_of_the_reserved_sm_launch():
    """The 2048-problem N = 10 batch of the reserved-SM launch at default settings."""
    B, N = 2048, 10
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=41, mu=(0.3, 1.0))
    f = draw(B, N, seed=41)
    mpc = pkg.BatchedMPC(N=N, max_batch=B)
    put(mpc, f)
    check_solved(mpc, pb, f, run(mpc, pb))
