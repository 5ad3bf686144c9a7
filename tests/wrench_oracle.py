"""fp64 statement of the per-robot external wrench (cmpc_set_wrench) for the tests, independent of the shift the
library applies: a known force F_j and torque tau_j (world frame) at stage j is the affine term dt E_j of the
sparse-form dynamics,

    x_{j+1} = Ad x_j + dt B_j u_j + dt E_j,   E_j = [0, 0, Ihat^-1 tau_j, F_j / m, 0],   Ihat^-1 = Rz Ib^-1 Rz',

so that the condensed QP keeps body_oracle's prediction matrix and c0 becomes the free response of x0 plus the
response to that term.  Everything else is body_oracle's (and through it condensed_admm's and tight_ipm's); the
contact oracle composes with ``condensed_qp`` below as it does with body_oracle's.
"""
import numpy as np

from oracle import condensed_admm as ca, srbd_qp, tight_ipm as ipm
import body_oracle as bo


def affine_term(x0, force, torque, mass=srbd_qp.MASS, ibody_inv=srbd_qp.IBODY_INV):
    """E (N,13): the continuous-time affine term of each stage."""
    Rz = srbd_qp.rot_z(x0[2])
    Ihat = Rz @ bo.ibody_inv_matrix(ibody_inv) @ Rz.T
    force, torque = np.asarray(force, dtype=float), np.asarray(torque, dtype=float)
    E = np.zeros((force.shape[0], 13))
    E[:, 6:9] = torque @ Ihat.T
    E[:, 9:12] = force / mass
    return E


def free_response(x0, force, torque, delta, mass=srbd_qp.MASS, ibody_inv=srbd_qp.IBODY_INV):
    """c0 (13,N+1): the trajectory with zero leg forces under the wrench, by the plain recursion."""
    E = affine_term(x0, force, torque, mass, ibody_inv)
    N = E.shape[0]
    Ad = np.eye(13) + delta * srbd_qp.continuous_A(x0[2])
    c0 = np.zeros((13, N + 1))
    c0[:, 0] = x0
    for k in range(N):
        c0[:, k + 1] = Ad @ c0[:, k] + delta * E[k]
    return c0


def condensed_qp(x0, r, stance, x_des, delta, force, torque, w=srbd_qp.W_STATE, mass=srbd_qp.MASS,
                 ibody_inv=srbd_qp.IBODY_INV, r_weight=0.0):
    """body_oracle.condensed_qp under the wrench: (H, g, S_c, c0, idx)."""
    N = r.shape[0]
    idx = srbd_qp.stance_index(stance)
    colsel = np.array([12 * i + 3 * l + k for (i, l) in idx for k in range(3)], dtype=int)
    S = bo.prediction_matrix(x0, r, delta, mass, ibody_inv)
    Sc = S[:, colsel] if len(colsel) else np.zeros((13 * (N + 1), 0))
    c0 = free_response(x0, force, torque, delta, mass, ibody_inv)
    Qbar = np.tile(w, N + 1)
    e0 = (c0 - x_des).T.reshape(-1)
    H = 2.0 * Sc.T @ (Qbar[:, None] * Sc) + 2.0 * r_weight * np.eye(len(colsel))
    gvec = 2.0 * Sc.T @ (Qbar * e0)
    return H, gvec, Sc, c0, idx


def admm_solve(x0, r, stance, x_des, mu, delta, force, torque, mass=srbd_qp.MASS, ibody_inv=srbd_qp.IBODY_INV,
               **kw):
    """condensed_admm.admm on the wrench QP; X includes the wrench's response."""
    H, g, Sc, c0, idx = condensed_qp(x0, r, stance, x_des, delta, force, torque, mass=mass, ibody_inv=ibody_inv)
    return bo._finish(ca.admm(H, g, mu, **kw), r, x_des, Sc, c0, idx, H, g)


def ipm_solve(x0, r, stance, x_des, mu, delta, force, torque, mass=srbd_qp.MASS, ibody_inv=srbd_qp.IBODY_INV,
              **kw):
    """tight_ipm.solve_qp on the wrench QP."""
    H, g, Sc, c0, idx = condensed_qp(x0, r, stance, x_des, delta, force, torque, mass=mass, ibody_inv=ibody_inv)
    return bo._finish(ipm.solve_qp(H, g, mu, **kw), r, x_des, Sc, c0, idx, H, g)
