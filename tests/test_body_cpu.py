"""Per-robot bodies without a GPU: the tests' full-inertia restatement of the oracle (body_oracle.py) and the
C ABI's argument checks."""
import ctypes as C

import numpy as np

import mpc_b200 as pkg
from mpc_b200.problems import synthetic_batch, random_bodies, DT
from oracle import condensed_admm as ca, srbd_qp, tight_ipm as ipm, wrench_form as wf
import body_oracle as bo


def test_body_oracle_with_a_diagonal_inertia_is_the_oracle_exactly():
    """The tests' full-inertia restatement (tests/body_oracle.py), given a diagonal inverse inertia as a 3x3
    matrix, reproduces the oracle's diagonal path bit for bit: the QP, the wrench map and the solves."""
    pb = synthetic_batch(4, N=10, gaits=pkg.problems.GAIT_NAMES, seed=6)
    ib = np.array([1 / 0.3, 1.2, 0.9])
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        a = srbd_qp.condensed_qp(x0, r, st, xd, DT, mass=7.5, ibody_inv=ib)
        m = bo.condensed_qp(x0, r, st, xd, DT, mass=7.5, ibody_inv=np.diag(ib))
        assert all(np.array_equal(u, v) for u, v in zip(a[:4], m[:4])) and a[4] == m[4]
        assert np.array_equal(srbd_qp.continuous_B(x0[2], r[0], 7.5, ib), bo.continuous_B(x0[2], r[0], 7.5, np.diag(ib)))
        assert np.array_equal(wf.leg_maps(x0, r, ibody_inv=ib), bo.leg_maps(x0, r, np.diag(ib)))
        # the reference's body (the only one wrench_form.G_matrix takes) through both paths
        assert np.array_equal(wf.G_matrix(x0, r, st), bo.G_matrix(x0, r, st, ibody_inv=np.diag(srbd_qp.IBODY_INV)))
        ref = ca.solve_problem(x0, r, st, xd, mu, DT, fixed_iters=30, rho=0.5)
        got = bo.admm_solve(x0, r, st, xd, mu, DT, srbd_qp.MASS, srbd_qp.IBODY_INV, fixed_iters=30, rho=0.5)
        assert np.array_equal(ref["U"], got["U"]) and ref["J"] == got["J"]
        if b == 0:
            ref = ipm.solve_problem(x0, r, st, xd, mu, DT)
            got = bo.ipm_solve(x0, r, st, xd, mu, DT, srbd_qp.MASS, np.diag(srbd_qp.IBODY_INV))
            assert np.array_equal(ref["U"], got["U"]) and ref["J"] == got["J"]


def test_random_bodies_are_physical_and_leave_other_draws_alone():
    before = synthetic_batch(8, N=10, seed=3).f32()
    mass, ib = random_bodies(256, seed=3)
    after = synthetic_batch(8, N=10, seed=3).f32()
    assert all(np.array_equal(a, b) for a, b in zip(before, after))
    assert mass.shape == (256,) and ib.shape == (256, 3, 3) and mass.dtype == ib.dtype == np.float64
    assert np.all((mass >= 0.75 * 8.885) & (mass <= 1.35 * 8.885))
    assert np.array_equal(ib, np.transpose(ib, (0, 2, 1)))
    assert np.all(np.linalg.eigvalsh(ib) > 0)
    inertia = np.sort(1.0 / np.linalg.eigvalsh(ib), axis=1)        # principal inertias
    assert np.all(inertia >= 0.7 * 0.24 - 1e-12) and np.all(inertia <= 1.4 * 1.0 + 1e-12)
    assert np.abs(ib[:, 0, 1]).max() > 1e-2                         # tilted axes: products of inertia
    m2, ib2 = random_bodies(256, seed=3)
    assert np.array_equal(mass, m2) and np.array_equal(ib, ib2)


def test_wrench_factorisation_holds_for_any_body():
    """H = G' M G with M built from the weights and dt alone: the body enters through G only."""
    pb = synthetic_batch(6, N=10, gaits=pkg.problems.GAIT_NAMES, seed=9)
    mass, ibs = random_bodies(pb.B, seed=9)
    M = wf.M_full(10, DT)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        H = bo.condensed_qp(x0, r, st, xd, DT, mass=mass[b], ibody_inv=ibs[b])[0]
        G = bo.G_matrix(x0, r, st, mass[b], ibs[b])
        assert np.abs(H - G.T @ M @ G).max() <= 1e-11 * max(np.abs(H).max(), 1.0)
        # and the body does change H
        assert np.abs(H - srbd_qp.condensed_qp(x0, r, st, xd, DT)[0]).max() > 1e-3 * np.abs(H).max()


def test_set_body_rejects_bad_arguments_without_a_device():
    L = pkg._capi.lib()
    assert "cmpc_set_body" in pkg._capi.SYMBOLS
    buf = (C.c_float * 16)()
    p = C.cast(buf, C.c_void_p)
    for args in ((None, 4, 0, p, p, None), (None, 0, 0, None, None, None), (None, -1, 0, p, p, None)):
        assert L.cmpc_set_body(*args) == -1             # CMPC_ERR_INVALID
        assert L.cmpc_last_error()
