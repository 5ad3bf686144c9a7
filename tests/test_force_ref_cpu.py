"""Per-robot force references without a GPU: the oracle's condensed terms against a direct evaluation of the
objective, the uniform-weight identity with r_weight, the generator, and the C ABI's argument checks."""
import ctypes as C

import numpy as np
import pytest

import mpc_b200 as pkg
from mpc_b200.problems import (synthetic_batch, random_bodies, random_contacts, random_weights, random_wrenches,
                               random_force_refs, DT, GAIT_NAMES)
from oracle import srbd_qp
import body_oracle as bo
import force_ref_oracle as fo


def direct_objective(x0, r, stance, xd, u, Sc, c0, idx, w, r_weight, f_ref, weight):
    """the objective of the force vector u (stacked stance forces) from simulated states"""
    N = r.shape[0]
    X = c0 + (Sc @ u).reshape(N + 1, 13).T
    J = srbd_qp.objective(X, xd, w) + r_weight * float(u @ u)
    for s, (i, l) in enumerate(idx):
        J += weight[i, l] * float(np.sum((u[3 * s:3 * s + 3] - f_ref[i, l]) ** 2))
    return J


@pytest.mark.parametrize("N", [1, 4, 10, 30])
def test_condensed_terms_match_the_objective(N):
    pb = synthetic_batch(5, N=N, gaits=GAIT_NAMES, seed=N)
    w, rw = random_weights(pb.B, seed=N)
    m, ib = random_bodies(pb.B, seed=N)
    f_ref, weight = random_force_refs(pb.B, N, seed=N)
    weight = weight * 1e3                                    # large enough to dominate a difference
    rng = np.random.default_rng(N)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        kw = dict(w=w[b], r_weight=rw[b], mass=m[b], ibody_inv=ib[b])
        H, g, Sc, c0, idx = fo.condensed_qp(x0, r, st, xd, DT, f_ref[b], weight[b], **kw)
        if not len(idx):
            continue
        q = lambda u: 0.5 * u @ H @ u + g @ u
        J = lambda u: direct_objective(x0, r, st, xd, u, Sc, c0, idx, w[b], rw[b], f_ref[b], weight[b])
        u0 = rng.normal(0.0, 30.0, H.shape[0])
        for _ in range(3):
            u1 = rng.normal(0.0, 30.0, H.shape[0])
            dj, dq = J(u1) - J(u0), q(u1) - q(u0)
            assert abs(dj - dq) <= 1e-9 * max(abs(J(u1)), abs(J(u0)), 1.0), (b, dj, dq)


def test_uniform_weight_with_zero_reference_is_r_weight():
    pb = synthetic_batch(4, N=10, gaits=GAIT_NAMES, seed=5)
    c = 3e-3
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        a = fo.condensed_qp(x0, r, st, xd, DT, np.zeros((10, 4, 3)), np.full((10, 4), c), r_weight=1e-4)
        ref = bo.condensed_qp(x0, r, st, xd, DT, r_weight=1e-4 + c)
        assert np.abs(a[0] - ref[0]).max() <= 1e-12 * np.abs(ref[0]).max()
        assert np.array_equal(a[1], ref[1])


def test_zero_weight_is_the_plain_qp():
    pb = synthetic_batch(4, N=10, gaits=GAIT_NAMES, seed=6)
    f_ref, _ = random_force_refs(pb.B, 10, seed=6)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        a = fo.condensed_qp(x0, r, st, xd, DT, f_ref[b], np.zeros((10, 4)))
        ref = bo.condensed_qp(x0, r, st, xd, DT)
        for x, y in zip(a[:4], ref[:4]):
            assert np.array_equal(x, y)


def test_random_force_refs_are_deterministic_and_leave_other_draws_alone():
    B, N = 64, 10
    before = (synthetic_batch(8, N=N, seed=3).f32(), random_bodies(8, seed=3), random_contacts(8, N, seed=3),
              random_weights(8, seed=3), random_wrenches(8, N, seed=3))
    f, w = random_force_refs(B, N, seed=3)
    after = (synthetic_batch(8, N=N, seed=3).f32(), random_bodies(8, seed=3), random_contacts(8, N, seed=3),
             random_weights(8, seed=3), random_wrenches(8, N, seed=3))
    for x, y in zip(before, after):
        assert all(np.array_equal(a, b) for a, b in zip(x, y))
    f2, w2 = random_force_refs(B, N, seed=3)
    assert np.array_equal(f, f2) and np.array_equal(w, w2)
    assert not np.array_equal(f, random_force_refs(B, N, seed=4)[0])
    assert f.shape == (B, N, 4, 3) and w.shape == (B, N, 4) and f.dtype == w.dtype == np.float64
    mg = pkg.problems.REF_MASS * 9.81
    assert np.all(np.abs(f[..., :2]) <= 0.1 * mg) and np.all((f[..., 2] >= 0.4 * mg) & (f[..., 2] <= 0.6 * mg))
    assert np.all((w >= 1e-4) & (w <= 1e-2))
    assert np.all(f[0::2] == f[0::2, :1]) and np.all(w[0::2] == w[0::2, :1])     # one per leg for the horizon


def test_set_force_ref_rejects_bad_arguments_without_a_device():
    L = pkg._capi.lib()
    assert "cmpc_set_force_ref" in pkg._capi.SYMBOLS
    buf = (C.c_float * 16)()
    p = C.cast(buf, C.c_void_p)
    for args in ((None, 4, 0, p, p, None), (None, 0, 0, None, None, None), (None, -1, 0, p, p, None)):
        assert L.cmpc_set_force_ref(*args) == -1          # CMPC_ERR_INVALID
        assert L.cmpc_last_error()
