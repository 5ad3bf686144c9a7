"""The composed per-slot oracle (mix_oracle.py) without a GPU: with every feature at its default it is the oracle's
ADMM, and restricted to one feature it is that feature's own oracle, at fixed iteration counts to 1e-10."""
import numpy as np
import pytest

from mpc_b200.problems import (synthetic_batch, random_bodies, random_contacts, random_weights, random_wrenches, DT,
                               GAIT_NAMES)
from oracle import condensed_admm as ca
import body_oracle as bo
import contact_oracle as co
import wrench_oracle as wo
import mix_oracle as mo

K = 40
KW = dict(fixed_iters=K, rho=0.5)


def draw(B, N, seed):
    m, ib = random_bodies(B, seed=seed)
    normal, mu, lo, hi = random_contacts(B, N, seed=seed)
    w, rw = random_weights(B, seed=seed)
    force, torque = random_wrenches(B, N, seed=seed)
    f = dict(mass=m, ibody_inv=ib, normal=normal, mu=mu, f_min=lo, f_max=hi, w=w, r_weight=rw, force=force,
             torque=torque)
    return {k: mo.r32(v) for k, v in f.items()}


def close(a, b):
    return np.abs(a - b).max() <= 1e-10 * max(1.0, np.abs(b).max())


def same_solve(got, ref):
    return close(got["U"], ref["U"]) and close(got["X"], ref["X"]) and close(got["y"], ref["y"])


@pytest.mark.parametrize("N", [5, 10])
def test_defaults_are_the_oracle(N):
    pb = synthetic_batch(4, N=N, gaits=GAIT_NAMES, seed=N)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        ref = ca.solve_problem(x0, r, st, xd, mu, DT, **KW)
        assert same_solve(mo.mix_admm(pb, b, {}, **KW), ref), b


@pytest.mark.parametrize("N", [5, 10])
def test_each_feature_alone_is_its_own_oracle(N):
    pb = synthetic_batch(4, N=N, gaits=GAIT_NAMES, seed=N)
    f = draw(pb.B, N, seed=N)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        body = {k: f[k] for k in ("mass", "ibody_inv")}
        ref = bo.admm_solve(x0, r, st, xd, mu, DT, f["mass"][b], f["ibody_inv"][b], **KW)
        assert same_solve(mo.mix_admm(pb, b, body, **KW), ref), (b, "body")
        contact = {k: f[k] for k in ("normal", "mu", "f_min", "f_max")}
        ref = co.admm_solve(x0, r, st, xd, DT, f["normal"][b], f["mu"][b], f["f_min"][b], f["f_max"][b], **KW)
        assert same_solve(mo.mix_admm(pb, b, contact, **KW), ref), (b, "contact")
        H, g, Sc, c0, idx = bo.condensed_qp(x0, r, st, xd, DT, w=f["w"][b], r_weight=f["r_weight"][b])
        ref = bo._finish(ca.admm(H, g, mu, **KW), r, xd, Sc, c0, idx, H, g)
        assert same_solve(mo.mix_admm(pb, b, {k: f[k] for k in ("w", "r_weight")}, **KW), ref), (b, "weights")
        ref = wo.admm_solve(x0, r, st, xd, mu, DT, f["force"][b], f["torque"][b], **KW)
        assert same_solve(mo.mix_admm(pb, b, {k: f[k] for k in ("force", "torque")}, **KW), ref), (b, "wrench")


def test_all_features_compose():
    """With all four groups the QP is wrench_oracle's with the slot's body and weights, every feature moves the
    solution, and the projection keeps each stance force in its own surface's frustum."""
    N = 10
    pb = synthetic_batch(4, N=N, gaits=GAIT_NAMES, seed=2)
    f = draw(pb.B, N, seed=2)
    for b in range(pb.B):
        x0, r, st, xd, mu = pb.problem(b)
        H, g, Sc, c0, idx, legs = mo.mix_qp(pb, b, f)
        Hw, gw, _, c0w, _ = wo.condensed_qp(x0, r, st, xd, DT, f["force"][b], f["torque"][b], w=f["w"][b],
                                            mass=f["mass"][b], ibody_inv=f["ibody_inv"][b], r_weight=f["r_weight"][b])
        assert np.array_equal(H, Hw) and np.array_equal(g, gw) and np.array_equal(c0, c0w)
        full = mo.mix_admm(pb, b, f, **KW)
        for drop in (("mass", "ibody_inv"), ("normal", "mu", "f_min", "f_max"), ("w",), ("force", "torque")):
            part = mo.mix_admm(pb, b, {k: v for k, v in f.items() if k not in drop}, **KW)
            assert np.abs(part["U"] - full["U"]).max() > 1e-3, (b, drop)
        z = full["z"].reshape(-1, 3)
        R, mu_l, lo, hi = legs
        loc = np.einsum("lki,lk->li", R, z)                                  # R' z per stance leg-stage
        tol = 1e-9 * (1.0 + np.abs(z).max())
        assert np.all(loc[:, 2] >= lo - tol) and np.all(loc[:, 2] <= hi + tol)
        assert np.all(np.abs(loc[:, :2]) <= mu_l[:, None] * loc[:, 2:] + tol)
        assert np.array_equal(mo.project(full["z"], legs).round(9), full["z"].round(9))
