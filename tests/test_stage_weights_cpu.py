"""Per-robot stage weights without a GPU: the wrench-space factorisation with per-stage Gram matrices, the linear term
against a direct evaluation of the objective, the reduction of uniform stage weights to the weights oracle, the
generator, and the C ABI's argument checks."""
import ctypes as C

import numpy as np
import pytest

import mpc_b200 as pkg
from mpc_b200.problems import (synthetic_batch, random_bodies, random_contacts, random_weights, random_wrenches,
                               random_force_refs, random_stage_weights, REF_WEIGHTS, DT, GAIT_NAMES)
from oracle import srbd_qp, wrench_form as wf
import body_oracle as bo
import stage_weight_oracle as so


@pytest.mark.parametrize("N", [4, 10, 30])
def test_wrench_factorisation_holds_for_stage_weights(N):
    """H = G' M G + 2 r_weight I in fp64 with M_a of the per-stage formula, against Sc' Qbar Sc of the oracle, for
    every kind of random_stage_weights and a random body: the stage weights enter H through M only."""
    pb = synthetic_batch(8, N=N, gaits=GAIT_NAMES, seed=N)
    ws = random_stage_weights(pb.B, N, seed=N)
    m, ib = random_bodies(pb.B, seed=N)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        rw = 1e-4 * (b % 2)
        H = so.condensed_qp(x0, r, st, xd, DT, ws[b], mass=m[b], ibody_inv=ib[b], r_weight=rw)[0]
        Ma = so.axis_gram(DT, ws[b])
        M = np.zeros((6 * N, 6 * N))
        for a in range(6):
            M[a::6, a::6] = Ma[a]
        G = bo.G_matrix(x0, r, st, m[b], ib[b])
        want = G.T @ M @ G + 2.0 * rw * np.eye(G.shape[1])
        assert np.abs(H - want).max() <= 1e-11 * max(np.abs(H).max(), 1.0), b
    # the per-stage formula is wrench_form's with the same row on every stage
    w = REF_WEIGHTS
    assert np.abs(so.axis_gram(DT, np.tile(w, (N, 1))) - wf.axis_gram(N, DT, w)).max() <= \
        1e-14 * np.abs(wf.axis_gram(N, DT, w)).max()


@pytest.mark.parametrize("N", [1, 5, 10, 30])
def test_linear_term_matches_the_objective(N):
    """g (and H) against a direct evaluation of the objective from simulated states, with a wrench: differences of
    J between random force vectors equal those of the quadratic model."""
    pb = synthetic_batch(6, N=N, gaits=GAIT_NAMES, seed=20 + N)
    ws = random_stage_weights(pb.B, N, seed=20 + N)
    force, torque = random_wrenches(pb.B, N, seed=N)
    rng = np.random.default_rng(N)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        H, g, Sc, c0, idx = so.condensed_qp(x0, r, st, xd, DT, ws[b], force[b], torque[b], r_weight=1e-4)
        if not len(idx):
            continue
        q = lambda u: 0.5 * u @ H @ u + g @ u

        def J(u):
            X = c0 + (Sc @ u).reshape(N + 1, 13).T
            return so.objective(X, xd, ws[b]) + 1e-4 * float(u @ u)
        u0 = rng.normal(0.0, 30.0, H.shape[0])
        for _ in range(3):
            u1 = rng.normal(0.0, 30.0, H.shape[0])
            dj, dq = J(u1) - J(u0), q(u1) - q(u0)
            assert abs(dj - dq) <= 1e-9 * max(abs(J(u1)), abs(J(u0)), 1.0), (b, dj, dq)


def test_uniform_stage_weights_are_the_weights_oracle():
    """the same row on every stage gives body_oracle's QP (one row tiled) exactly"""
    pb = synthetic_batch(6, N=10, gaits=GAIT_NAMES, seed=8)
    w, rw = random_weights(pb.B, seed=8)
    m, ib = random_bodies(pb.B, seed=8)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        kw = dict(mass=m[b], ibody_inv=ib[b], r_weight=rw[b])
        a = so.condensed_qp(x0, r, st, xd, DT, np.tile(w[b], (10, 1)), **kw)
        ref = bo.condensed_qp(x0, r, st, xd, DT, w=w[b], **kw)
        for x, y in zip(a[:4], ref[:4]):
            assert np.array_equal(x, y)


def test_terminal_weight_changes_only_the_last_stage_cost():
    """a heavier last row changes H and g, and leaves the objective of a trajectory that meets x_des at stage N alone"""
    pb = synthetic_batch(2, N=10, gaits=("trot",), seed=9)
    x0, r, st, xd, mu = pb.problem(0)
    w = np.tile(REF_WEIGHTS, (10, 1))
    wt = w.copy()
    wt[-1] *= 30.0
    a = so.condensed_qp(x0, r, st, xd, DT, w)
    t = so.condensed_qp(x0, r, st, xd, DT, wt)
    assert np.abs(t[0] - a[0]).max() > 1e-3 * np.abs(a[0]).max()
    X = xd.copy()
    X[:, :-1] += 1.0
    assert so.objective(X, xd, w) == so.objective(X, xd, wt)


def test_mix_oracle_without_stage_weights_is_the_force_ref_oracle():
    B, N = 4, 10
    pb = synthetic_batch(B, N=N, gaits=GAIT_NAMES, seed=2)
    f = {}
    f.update(zip(("mass", "ibody_inv"), random_bodies(B, seed=2)))
    f.update(zip(("normal", "mu", "f_min", "f_max"), random_contacts(B, N, seed=2)))
    f.update(zip(("w", "r_weight"), random_weights(B, seed=2)))
    f.update(zip(("force", "torque"), random_wrenches(B, N, seed=2)))
    f.update(zip(("f_ref", "f_weight"), random_force_refs(B, N, seed=2)))
    import force_ref_oracle as fo
    for b in range(B):
        a, ref = so.mix_qp(pb, b, f), fo.mix_qp(pb, b, f)
        assert np.array_equal(a[0], ref[0]) and np.array_equal(a[1], ref[1])
        # the slot's row on every stage: the same QP up to rounding of the wrench's free response
        g = dict(f, w_stage=np.repeat(f["w"][:, None, :], N, axis=1))
        s = so.mix_qp(pb, b, g)
        assert np.abs(s[0] - ref[0]).max() <= 1e-12 * np.abs(ref[0]).max()
        assert np.abs(s[1] - ref[1]).max() <= 1e-9 * max(np.abs(ref[1]).max(), 1.0)


def test_random_stage_weights_are_deterministic_valid_and_leave_other_draws_alone():
    B, N = 64, 10
    before = (synthetic_batch(8, N=N, seed=3).f32(), random_bodies(8, seed=3), random_weights(8, seed=3),
              random_force_refs(8, N, seed=3))
    w = random_stage_weights(B, N, seed=3)
    after = (synthetic_batch(8, N=N, seed=3).f32(), random_bodies(8, seed=3), random_weights(8, seed=3),
             random_force_refs(8, N, seed=3))
    for x, y in zip(before, after):
        assert all(np.array_equal(a, b) for a, b in zip(x, y))
    assert np.array_equal(w, random_stage_weights(B, N, seed=3))
    assert not np.array_equal(w, random_stage_weights(B, N, seed=4))
    assert w.shape == (B, N, 13) and w.dtype == np.float64
    # the validity rules of cmpc_set_stage_weights, on every stage
    assert np.all(np.isfinite(w)) and np.all(w >= 0) and np.all(w[..., 6] == w[..., 7]) and np.all(w[..., 12] == 0)
    assert np.all(w[..., 6:12] > 0)
    f = w[..., :12] / REF_WEIGHTS[:12]
    assert np.all(w[0::4] == w[0::4, :1])                                   # one row for the horizon
    assert np.all((f[0::4] >= 0.25 * (1 - 1e-12)) & (f[0::4] <= 4.0 * (1 + 1e-12)))
    assert np.all(f[1::4, :-1] == 1.0) and np.all((f[1::4, -1] >= 1.0) & (f[1::4, -1] <= 30.0 * (1 + 1e-12)))
    assert np.allclose(f[2::8, 0], 0.25) and np.allclose(f[2::8, -1], 1.0)   # ramps, rising and falling
    assert np.allclose(f[6::8, 0], 1.0) and np.allclose(f[6::8, -1], 0.25)
    zero = np.all(w[3::4, :, :6] == 0, axis=2)
    assert np.all(zero.any(axis=1)) and not zero[:, -1].any()             # a window, never the last stage


def test_set_stage_weights_rejects_bad_arguments_without_a_device():
    L = pkg._capi.lib()
    assert "cmpc_set_stage_weights" in pkg._capi.SYMBOLS
    buf = (C.c_float * 16)()
    p = C.cast(buf, C.c_void_p)
    for args in ((None, 4, 0, p, p, None), (None, 0, 0, None, None, None), (None, -1, 0, p, p, None)):
        assert L.cmpc_set_stage_weights(*args) == -1          # CMPC_ERR_INVALID
        assert L.cmpc_last_error()
