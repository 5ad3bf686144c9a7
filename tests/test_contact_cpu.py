"""Per-foot contact surfaces without a GPU: the contact frame, the rotated projection, the tests' restatement of the
oracle with per-leg surfaces (contact_oracle.py), random_contacts and the C ABI's argument checks."""
import ctypes as C

import numpy as np

import mpc_b200 as pkg
from mpc_b200.problems import synthetic_batch, random_bodies, random_contacts, DT
from oracle import condensed_admm as ca, srbd_qp, tight_ipm as ipm
import contact_oracle as co


def test_contact_frame_is_orthonormal_right_handed_and_identity_on_flat_ground():
    rng = np.random.default_rng(0)
    normals = np.concatenate([rng.normal(size=(500, 3)), [[1, 0, 0], [-3, 0, 0], [0, 1, 0], [1, 1, 0], [1, 0, 1e-3]]])
    R = co.contact_frame(normals)
    assert np.abs(np.einsum("bki,bkj->bij", R, R) - np.eye(3)).max() < 1e-12
    assert np.abs(np.linalg.det(R) - 1.0).max() < 1e-12
    assert np.abs(R[:, :, 2] - normals / np.linalg.norm(normals, axis=1, keepdims=True)).max() < 1e-15
    nx2 = (normals[:, 0] / np.linalg.norm(normals, axis=1)) ** 2
    assert (nx2 <= 0.5).any() and (nx2 > 0.5).any()                        # both branches of the rule
    # t1 lies in the plane of n and its basis vector: e_x on the first branch, e_y on the second
    t1, n = R[:, :, 0], R[:, :, 2]
    e = np.where((nx2 <= 0.5)[:, None], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0])
    assert np.abs(np.einsum("bi,bi->b", np.cross(e, n), t1)).max() < 1e-12
    for c in (1.0, 2.5):
        assert np.array_equal(co.contact_frame(np.array([0.0, 0.0, c])), np.eye(3))
        assert np.array_equal(co.contact_frame(np.array([0.0, 0.0, c], dtype=np.float32).astype(np.float64)), np.eye(3))


def test_rotated_projection_is_the_euclidean_projection():
    rng = np.random.default_rng(1)
    for _ in range(40):
        R = co.contact_frame(rng.normal(size=3))
        mu = rng.uniform(0.0, 1.2)
        lo = rng.uniform(0.0, 10.0)
        hi = lo + rng.uniform(0.0, 80.0)
        w = rng.normal(0, 60.0, size=(200, 3))
        p = co.project(w, np.broadcast_to(R, (200, 3, 3)), mu, lo, hi)
        loc = p @ R                                                      # R' p per row
        tol = 1e-9 * (1.0 + np.abs(w).max())
        assert np.all(loc[:, 2] >= lo - tol) and np.all(loc[:, 2] <= hi + tol)
        assert np.all(np.abs(loc[:, 0]) <= mu * loc[:, 2] + tol) and np.all(np.abs(loc[:, 1]) <= mu * loc[:, 2] + tol)
        # random feasible points q: the variational inequality of the projection, (w - p).(q - p) <= 0
        fz = rng.uniform(lo, hi, 300)
        q = np.stack([rng.uniform(-1, 1, 300) * mu * fz, rng.uniform(-1, 1, 300) * mu * fz, fz], 1) @ R.T
        assert np.all(np.einsum("bi,qbi->qb", w - p, q[:, None, :] - p[None]) <= 1e-9 * (1.0 + np.abs(w).max() ** 2))
        assert np.array_equal(co.project(p, np.broadcast_to(R, (200, 3, 3)), mu, lo, hi).round(9), p.round(9))


def test_contact_oracle_on_flat_ground_is_the_oracle_exactly():
    """Flat normals (any length) with the problem's mu and the default bounds reproduce the oracle's ADMM and
    interior-point solves bit for bit."""
    pb = synthetic_batch(4, N=10, gaits=pkg.problems.GAIT_NAMES, seed=6)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        normal = np.tile([0.0, 0.0, 2.5 if b % 2 else 1.0], (10, 4, 1))
        mus = np.full((10, 4), mu)
        lo, hi = np.full((10, 4), srbd_qp.F_MIN), np.full((10, 4), srbd_qp.F_MAX)
        ref = ca.solve_problem(x0, r, st, xd, mu, DT, fixed_iters=30, rho=0.5)
        got = co.admm_solve(x0, r, st, xd, DT, normal, mus, lo, hi, fixed_iters=30, rho=0.5)
        assert np.array_equal(ref["U"], got["U"]) and ref["J"] == got["J"]
        ref = ca.solve_problem(x0, r, st, xd, mu, DT, rho=0.5, adaptive_interval=25)
        got = co.admm_solve(x0, r, st, xd, DT, normal, mus, lo, hi, rho=0.5, adaptive_interval=25)
        assert np.array_equal(ref["U"], got["U"]) and ref["iters"] == got["iters"]
        if b < 2:
            ref = ipm.solve_problem(x0, r, st, xd, mu, DT)
            got = co.ipm_solve(x0, r, st, xd, DT, normal, mus, lo, hi)
            assert np.array_equal(ref["U"], got["U"]) and ref["J"] == got["J"]


def test_ipm_with_random_contacts_is_feasible_in_each_legs_frame():
    N = 10
    pb = synthetic_batch(3, N=N, gaits=pkg.problems.GAIT_NAMES, seed=4)
    normal, mu, lo, hi = random_contacts(pb.B, N, seed=4)
    mass, ibs = random_bodies(pb.B, seed=4)
    for b in range(pb.B):
        x0, r, st, xd, _ = pb.problem(b)
        kw = dict(mass=mass[b], ibody_inv=ibs[b]) if b == 2 else {}            # bodies and contacts compose
        out = co.ipm_solve(x0, r, st, xd, DT, normal[b], mu[b], lo[b], hi[b], **kw)
        assert out["res"] < 1e-6 * max(1.0, np.abs(out["g"]).max()) and out["gap"] < 1e-8
        R = co.contact_frame(normal[b])
        loc = np.einsum("jlki,jlk->jli", R, out["U"].reshape(N, 4, 3))        # R' f per leg-stage
        on = st.astype(bool)
        tol = 1e-7
        assert np.all(loc[on][:, 2] >= lo[b][on] - tol) and np.all(loc[on][:, 2] <= hi[b][on] + tol)
        assert np.all(np.abs(loc[on][:, :2]) <= mu[b][on][:, None] * loc[on][:, 2:] + tol)
        assert np.all(out["U"].reshape(N, 4, 3)[~on] == 0.0)
        # the surfaces matter: the flat-ground optimum is a different point
        flat = ipm.solve_problem(x0, r, st, xd, 0.6, DT)
        assert np.abs(flat["U"] - out["U"]).max() > 1e-2


def test_random_contacts_are_deterministic_and_leave_other_draws_alone():
    before = synthetic_batch(8, N=10, seed=3).f32()
    body = random_bodies(8, seed=3)
    normal, mu, lo, hi = random_contacts(64, 12, seed=3)
    after = synthetic_batch(8, N=10, seed=3).f32()
    assert all(np.array_equal(a, b) for a, b in zip(before, after))
    assert all(np.array_equal(a, b) for a, b in zip(body, random_bodies(8, seed=3)))
    again = random_contacts(64, 12, seed=3)
    assert all(np.array_equal(a, b) for a, b in zip((normal, mu, lo, hi), again))
    assert normal.shape == (64, 12, 4, 3) and mu.shape == lo.shape == hi.shape == (64, 12, 4)
    assert np.abs(np.linalg.norm(normal, axis=-1) - 1.0).max() < 1e-12
    tilt = np.degrees(np.arccos(normal[..., 2]))
    assert tilt.max() < 30.0 and tilt.mean(axis=(1, 2)).max() > 10.0      # inclines up to 20 deg, jittered
    assert np.all((mu >= 0.3) & (mu <= 1.0)) and np.all(lo == 3.0)
    assert np.all((hi >= 40.0) & (hi <= 100.0)) and np.all(hi == hi[:, :1])  # per leg, every stage
    assert not np.array_equal(random_contacts(64, 12, seed=4)[0], normal)


def test_set_contact_rejects_bad_arguments_without_a_device():
    L = pkg._capi.lib()
    assert "cmpc_set_contact" in pkg._capi.SYMBOLS
    buf = (C.c_float * 16)()
    p = C.cast(buf, C.c_void_p)
    for args in ((None, 4, 0, p, p, p, p, None), (None, 0, 0, None, None, None, None, None),
                 (None, -1, 0, p, p, p, p, None)):
        assert L.cmpc_set_contact(*args) == -1          # CMPC_ERR_INVALID
        assert L.cmpc_last_error()
