"""fp64 restatement of the per-robot body (cmpc_set_body) for the tests: the QP of one problem with its own
mass and a full 3x3 body-frame inverse inertia.

The oracle package (``oracle.srbd_qp`` and friends) models the reference's diagonal inertia only and stays as
it is; the functions here follow its code line for line with the inertia as a matrix, so a diagonal matrix
reproduces the oracle's numbers exactly (``tests/test_body_cpu.py`` checks that) and everything else reuses it.
"""
import numpy as np

from oracle import condensed_admm as ca, srbd_qp, tight_ipm as ipm


def ibody_inv_matrix(ibody_inv):
    """(3,) = the diagonal, as the reference writes it, or (3,3)."""
    ib = np.asarray(ibody_inv, dtype=float)
    return np.diag(ib) if ib.shape == (3,) else ib


def continuous_B(yaw, r_stage, mass=srbd_qp.MASS, ibody_inv=srbd_qp.IBODY_INV):
    """srbd_qp.continuous_B with a full inverse inertia."""
    Rz = srbd_qp.rot_z(yaw)
    I_hat_inv = Rz @ ibody_inv_matrix(ibody_inv) @ Rz.T
    B = np.zeros((13, 12))
    for l in range(4):
        B[6:9, 3 * l:3 * l + 3] = I_hat_inv @ srbd_qp.skew(r_stage[l])
        B[9:12, 3 * l:3 * l + 3] = np.eye(3) / mass
    return B


def prediction_matrix(x0, r, delta, mass=srbd_qp.MASS, ibody_inv=srbd_qp.IBODY_INV):
    N = r.shape[0]
    yaw = x0[2]
    Ad = np.eye(13) + delta * srbd_qp.continuous_A(yaw)
    S = np.zeros((13 * (N + 1), 12 * N))
    for j in range(N):
        blk = delta * continuous_B(yaw, r[j], mass, ibody_inv)
        for k in range(j + 1, N + 1):
            S[13 * k:13 * k + 13, 12 * j:12 * j + 12] = blk
            blk = Ad @ blk
    return S


def condensed_qp(x0, r, stance, x_des, delta, w=srbd_qp.W_STATE, mass=srbd_qp.MASS,
                 ibody_inv=srbd_qp.IBODY_INV, r_weight=0.0):
    """srbd_qp.condensed_qp with a full inverse inertia: (H, g, S_c, c0, idx)."""
    N = r.shape[0]
    idx = srbd_qp.stance_index(stance)
    colsel = np.array([12 * i + 3 * l + k for (i, l) in idx for k in range(3)], dtype=int)
    S = prediction_matrix(x0, r, delta, mass, ibody_inv)
    Sc = S[:, colsel] if len(colsel) else np.zeros((13 * (N + 1), 0))
    c0 = srbd_qp.free_response(x0, N, delta)
    Qbar = np.tile(w, N + 1)
    e0 = (c0 - x_des).T.reshape(-1)
    H = 2.0 * Sc.T @ (Qbar[:, None] * Sc) + 2.0 * r_weight * np.eye(len(colsel))
    gvec = 2.0 * Sc.T @ (Qbar * e0)
    return H, gvec, Sc, c0, idx


def leg_maps(x0, r, ibody_inv=srbd_qp.IBODY_INV):
    """wrench_form.leg_maps with a full inverse inertia: Ghat (N,4,3,3) = Rz I^-1_hat [r]x."""
    Rz = srbd_qp.rot_z(x0[2])
    Ihat = Rz @ ibody_inv_matrix(ibody_inv) @ Rz.T
    N = r.shape[0]
    Gh = np.zeros((N, 4, 3, 3))
    for j in range(N):
        for l in range(4):
            Gh[j, l] = Rz @ Ihat @ srbd_qp.skew(r[j, l])
    return Gh


def G_matrix(x0, r, stance, mass=srbd_qp.MASS, ibody_inv=srbd_qp.IBODY_INV):
    """wrench_form.G_matrix with the body: G (6N x n) on the compact stance unknowns."""
    N = r.shape[0]
    idx = srbd_qp.stance_index(stance)
    Gh = leg_maps(x0, r, ibody_inv)
    G = np.zeros((6 * N, 3 * len(idx)))
    for s, (j, l) in enumerate(idx):
        G[6 * j:6 * j + 3, 3 * s:3 * s + 3] = Gh[j, l]
        G[6 * j + 3:6 * j + 6, 3 * s:3 * s + 3] = np.eye(3) / mass
    return G


def _finish(info, r, x_des, Sc, c0, idx, H, gvec):
    N = r.shape[0]
    U = np.zeros((N, 12))
    for s, (i, l) in enumerate(idx):
        U[i, 3 * l:3 * l + 3] = info["x"][3 * s:3 * s + 3]
    X = c0 + (Sc @ info["x"]).reshape(N + 1, 13).T if len(idx) else c0
    info.update(U=U, X=X, J=srbd_qp.objective(X, x_des), wrench=srbd_qp.stage_wrench(U, r), H=H, g=gvec, idx=idx)
    return info


def admm_solve(x0, r, stance, x_des, mu, delta, mass, ibody_inv, **kw):
    """condensed_admm.solve_problem (r_weight = 0) for the given body."""
    H, gvec, Sc, c0, idx = condensed_qp(x0, r, stance, x_des, delta, mass=mass, ibody_inv=ibody_inv)
    return _finish(ca.admm(H, gvec, mu, **kw), r, x_des, Sc, c0, idx, H, gvec)


def ipm_solve(x0, r, stance, x_des, mu, delta, mass, ibody_inv, **kw):
    """tight_ipm.solve_problem (r_weight = 0) for the given body."""
    H, gvec, Sc, c0, idx = condensed_qp(x0, r, stance, x_des, delta, mass=mass, ibody_inv=ibody_inv)
    return _finish(ipm.solve_qp(H, gvec, mu, **kw), r, x_des, Sc, c0, idx, H, gvec)
