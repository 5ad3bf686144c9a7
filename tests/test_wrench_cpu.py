"""Per-robot external wrench without a GPU: the identity the library's shift rests on (the QP under a known wrench is
the QP without it on x_des - phi, and its X is that QP's X + phi), the wrench generator and the C ABI's argument
checks."""
import ctypes as C

import numpy as np
import pytest

import mpc_b200 as pkg
from mpc_b200.problems import synthetic_batch, random_bodies, random_contacts, random_weights, random_wrenches, DT
from oracle import srbd_qp
import body_oracle as bo
import wrench_oracle as wo


def phi(x0, force, torque, delta, mass, ibody_inv):
    """(13,N+1) forced response of the wrench, restated from the formulas of cmpc_kernels.cuh (wrench_response):
    wrench axes [Rz (Rz Ib^-1 Rz') tau ; F / m], c1[k] = sum_{j<k}, c2[k] = sum_{j<k} (k-1-j);
    Theta += d^2 c2_ang, p += d^2 c2_lin, omega += d Rz' c1_ang, v += d c1_lin."""
    N = force.shape[0]
    Rz = srbd_qp.rot_z(x0[2])
    ib = bo.ibody_inv_matrix(ibody_inv)
    wv = np.concatenate([torque @ (Rz @ Rz @ ib @ Rz.T).T, force / mass], 1)    # (N,6)
    out = np.zeros((13, N + 1))
    for k in range(N + 1):
        c1 = wv[:k].sum(0)
        c2 = ((k - 1 - np.arange(k))[:, None] * wv[:k]).sum(0)
        out[0:3, k] = delta ** 2 * c2[:3]
        out[3:6, k] = delta ** 2 * c2[3:]
        out[6:9, k] = delta * Rz.T @ c1[:3]
        out[9:12, k] = delta * c1[3:]
    return out


@pytest.mark.parametrize("N", [1, 4, 10, 30, 60])
def test_wrench_qp_is_the_plain_qp_on_shifted_x_des(N):
    pb = synthetic_batch(6, N=N, gaits=pkg.problems.GAIT_NAMES, seed=N)
    m, ib = random_bodies(pb.B, seed=N)
    force, torque = random_wrenches(pb.B, N, seed=N)
    rng = np.random.default_rng(N)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        x0 = x0.copy()
        x0[2] = rng.uniform(-np.pi, np.pi)                 # any yaw
        kw = dict(mass=m[b], ibody_inv=ib[b])
        H, g, Sc, c0, idx = wo.condensed_qp(x0, r, st, xd, DT, force[b], torque[b], **kw)
        P = phi(x0, force[b], torque[b], DT, m[b], ib[b])
        H0, g0, Sc0, c00, _ = bo.condensed_qp(x0, r, st, xd - P, DT, **kw)
        assert np.array_equal(H, H0)
        assert np.abs(g - g0).max() <= 1e-10 * max(np.abs(g).max(), 1.0)
        assert np.abs(c0 - (c00 + P)).max() <= 1e-12 * max(np.abs(c0).max(), 1.0)
        # X of any force vector: the wrench oracle's = the shifted QP's + phi
        u = rng.normal(0.0, 30.0, Sc.shape[1])
        X = c0 + (Sc @ u).reshape(N + 1, 13).T
        X0 = c00 + (Sc0 @ u).reshape(N + 1, 13).T
        assert np.abs(X - (X0 + P)).max() <= 1e-12 * max(np.abs(X).max(), 1.0)
        # and the wrench does move the QP
        if np.abs(force[b]).max() > 0 and len(idx):
            assert np.abs(g - bo.condensed_qp(x0, r, st, xd, DT, **kw)[1]).max() > 1e-6 * np.abs(g).max()


def test_zero_wrench_is_the_body_oracle():
    pb = synthetic_batch(4, N=10, seed=2)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        z = np.zeros((10, 3))
        a = wo.condensed_qp(x0, r, st, xd, DT, z, z)
        c = bo.condensed_qp(x0, r, st, xd, DT)
        for x, y in zip(a[:4], c[:4]):
            assert np.array_equal(x, y)


def test_random_wrenches_are_deterministic_and_leave_other_draws_alone():
    B, N = 256, 10
    before = (synthetic_batch(8, N=N, seed=3).f32(), random_bodies(8, seed=3), random_contacts(8, N, seed=3),
              random_weights(8, seed=3))
    f, t = random_wrenches(B, N, seed=3)
    after = (synthetic_batch(8, N=N, seed=3).f32(), random_bodies(8, seed=3), random_contacts(8, N, seed=3),
             random_weights(8, seed=3))
    for x, y in zip(before, after):
        assert all(np.array_equal(a, b) for a, b in zip(x, y))
    f2, t2 = random_wrenches(B, N, seed=3)
    assert np.array_equal(f, f2) and np.array_equal(t, t2)
    assert not np.array_equal(f, random_wrenches(B, N, seed=4)[0])
    assert f.shape == t.shape == (B, N, 3) and f.dtype == t.dtype == np.float64
    mg = pkg.problems.REF_MASS * 9.81
    assert np.all(np.hypot(f[..., 0], f[..., 1]) <= 0.2 * mg + 1e-9) and np.all(np.abs(f[..., 2]) <= 0.2 * mg + 1e-9)
    assert np.all(np.abs(t) <= 1.0)
    even, odd = f[0::2], f[1::2]
    assert np.all(even == even[:, :1]) and np.all(t[0::2] == t[0::2, :1])      # constant over the horizon
    assert np.all(t[1::2] == 0.0)
    on = np.any(odd != 0.0, axis=-1)                                          # the push: one window of stages
    for row in on:
        k = np.flatnonzero(row)
        assert 1 <= len(k) <= N // 2 and np.all(np.diff(k) == 1)


def test_set_wrench_rejects_bad_arguments_without_a_device():
    L = pkg._capi.lib()
    assert "cmpc_set_wrench" in pkg._capi.SYMBOLS
    buf = (C.c_float * 16)()
    p = C.cast(buf, C.c_void_p)
    for args in ((None, 4, 0, p, p, None), (None, 0, 0, None, None, None), (None, -1, 0, p, p, None)):
        assert L.cmpc_set_wrench(*args) == -1          # CMPC_ERR_INVALID
        assert L.cmpc_last_error()
