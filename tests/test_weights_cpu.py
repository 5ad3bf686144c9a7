"""Per-robot cost weights without a GPU: the wrench-space factorisation with any weights, the weight generator and the
C ABI's argument checks."""
import ctypes as C

import numpy as np

import mpc_b200 as pkg
from mpc_b200.problems import synthetic_batch, random_bodies, random_contacts, random_weights, REF_WEIGHTS, DT
from oracle import srbd_qp, wrench_form as wf
import body_oracle as bo


def test_wrench_factorisation_holds_for_any_weights():
    """H = G' M G + 2 r_weight I in fp64, with M = blockdiag of the per-axis Gram matrices of the problem's own
    weights (unequal axes, r_weight > 0 on odd problems): the weights enter through M and r_weight only."""
    pb = synthetic_batch(6, N=10, gaits=pkg.problems.GAIT_NAMES, seed=4)
    w, rw = random_weights(pb.B, seed=4)
    ib = np.diag(srbd_qp.IBODY_INV)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        H = bo.condensed_qp(x0, r, st, xd, DT, w=w[b], r_weight=rw[b])[0]
        assert np.array_equal(H, srbd_qp.condensed_qp(x0, r, st, xd, DT, w=w[b], r_weight=rw[b])[0])
        Ma = wf.axis_gram(10, DT, w[b])
        M = np.zeros((60, 60))
        for a in range(6):
            M[a::6, a::6] = Ma[a]
        G = bo.G_matrix(x0, r, st, srbd_qp.MASS, ib)
        want = G.T @ M @ G + 2.0 * rw[b] * np.eye(G.shape[1])
        assert np.abs(H - want).max() <= 1e-11 * max(np.abs(H).max(), 1.0)
        # and the weights do change H
        assert np.abs(H - srbd_qp.condensed_qp(x0, r, st, xd, DT)[0]).max() > 1e-2 * np.abs(H).max()


def test_random_weights_are_deterministic_valid_and_leave_other_draws_alone():
    before = synthetic_batch(8, N=10, seed=3).f32(), random_bodies(8, seed=3), random_contacts(8, 10, seed=3)
    w, rw = random_weights(256, seed=3)
    after = synthetic_batch(8, N=10, seed=3).f32(), random_bodies(8, seed=3), random_contacts(8, 10, seed=3)
    for x, y in zip(before, after):
        assert all(np.array_equal(a, b) for a, b in zip(x, y))
    w2, rw2 = random_weights(256, seed=3)
    assert np.array_equal(w, w2) and np.array_equal(rw, rw2)
    assert not np.array_equal(w, random_weights(256, seed=4)[0])
    assert w.shape == (256, 13) and rw.shape == (256,) and w.dtype == rw.dtype == np.float64
    # the validity rules of cmpc_set_weights
    assert np.all(np.isfinite(w)) and np.all(w >= 0) and np.all(w[:, 6] == w[:, 7]) and np.all(w[:, 12] == 0)
    assert np.all(w[:, 6:12] > 0)                          # every axis has a positive velocity-like weight
    f = w[:, :12] / REF_WEIGHTS[:12]
    assert np.all((f >= 0.25 * (1 - 1e-12)) & (f <= 4.0 * (1 + 1e-12)))
    assert np.log(f).std(axis=0).min() > 0.5               # spread over the whole range, per entry
    assert np.all(rw[0::2] == 0.0)
    assert np.all((rw[1::2] >= 1e-5 * (1 - 1e-12)) & (rw[1::2] <= 1e-2 * (1 + 1e-12)))


def test_set_weights_rejects_bad_arguments_without_a_device():
    L = pkg._capi.lib()
    assert "cmpc_set_weights" in pkg._capi.SYMBOLS
    buf = (C.c_float * 16)()
    p = C.cast(buf, C.c_void_p)
    for args in ((None, 4, 0, p, p, None), (None, 0, 0, None, None, None), (None, -1, 0, p, p, None)):
        assert L.cmpc_set_weights(*args) == -1          # CMPC_ERR_INVALID
        assert L.cmpc_last_error()
