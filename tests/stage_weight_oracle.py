"""fp64 statement of the per-robot stage weights (cmpc_set_stage_weights) for the tests: the state cost
sum_k (X_k - x_des_k)' diag(w_k) (X_k - x_des_k) with its own weights on every stage k = 1..N, i.e. the condensed
form of srbd_qp / body_oracle with Qbar built from an (N+1, 13) table of per-stage weights instead of one row tiled
N + 1 times.  Row 0 of that table weighs X_0 = x0, which the forces do not move: it has no effect on H or g.  The
stage weights w_stage (N, 13) of the library are rows 1..N (row i of w_stage weighs X_{i+1}).

``feats`` (mix_qp, mix_admm) is force_ref_oracle's dict with one more per-slot array: w_stage (B,N,13), which then
takes the place of w (r_weight stays); without it the problem keeps mix_oracle's one row of weights.
"""
import numpy as np

from oracle import srbd_qp
from mpc_b200.problems import DT
import body_oracle as bo
import contact_oracle as co
import force_ref_oracle as fo
import mix_oracle as mo
import wrench_oracle as wo


def stage_table(w_stage):
    """(N+1, 13) Qbar rows: w_stage (N, 13) below a row 0 (a copy of w_stage[0]; it multiplies zero rows of Sc)"""
    w_stage = np.asarray(w_stage, dtype=float)
    return np.vstack([w_stage[:1], w_stage])


def axis_gram(delta, w_stage):
    """M (6,N,N) of the stage weights: M_a[j][j'] = 2 sum_{k > max(j,j')} (w_pos,a,k d^4 (k-1-j)(k-1-j') +
    w_vel,a,k d^2), stage k's weights being w_stage[k-1] (wrench_form.axis_gram term by term)."""
    w_stage = np.asarray(w_stage, dtype=float)
    N = w_stage.shape[0]
    M = np.zeros((6, N, N))
    for a in range(6):
        for j in range(N):
            for jp in range(N):
                kk = np.arange(max(j, jp) + 1, N + 1)
                M[a, j, jp] = 2.0 * np.sum(w_stage[kk - 1, a] * delta ** 4 * (kk - 1 - j) * (kk - 1 - jp)
                                           + w_stage[kk - 1, 6 + a] * delta ** 2)
    return M


def condensed_qp(x0, r, stance, x_des, delta, w_stage, force=None, torque=None, mass=srbd_qp.MASS,
                 ibody_inv=srbd_qp.IBODY_INV, r_weight=0.0):
    """body_oracle.condensed_qp (wrench_oracle's with a wrench) with per-stage state weights: (H, g, S_c, c0, idx)"""
    N = r.shape[0]
    idx = srbd_qp.stance_index(stance)
    colsel = np.array([12 * i + 3 * l + k for (i, l) in idx for k in range(3)], dtype=int)
    S = bo.prediction_matrix(x0, r, delta, mass, ibody_inv)
    Sc = S[:, colsel] if len(colsel) else np.zeros((13 * (N + 1), 0))
    if force is None and torque is None:
        c0 = srbd_qp.free_response(x0, N, delta)
    else:
        z = np.zeros((N, 3))
        c0 = wo.free_response(x0, z if force is None else force, z if torque is None else torque, delta, mass,
                              ibody_inv)
    Qbar = stage_table(w_stage).reshape(-1)
    e0 = (c0 - x_des).T.reshape(-1)
    H = 2.0 * Sc.T @ (Qbar[:, None] * Sc) + 2.0 * r_weight * np.eye(len(colsel))
    gvec = 2.0 * Sc.T @ (Qbar * e0)
    return H, gvec, Sc, c0, idx


def objective(X, x_des, w_stage):
    """the state cost of the states X (13, N+1) over stages 1..N"""
    return float(np.sum(np.asarray(w_stage, dtype=float).T * (X[:, 1:] - x_des[:, 1:]) ** 2))


def mix_qp(pb, b, feats, delta=DT, as_f32=False):
    """force_ref_oracle.mix_qp with the slot's stage weights: (H, g, Sc, c0, idx, legs)"""
    if "w_stage" not in feats:
        return fo.mix_qp(pb, b, feats, delta, as_f32)
    x0, r, stance, xd, mu = mo.problem(pb, b, as_f32)
    f = mo.slot_features(feats, b, r.shape[0], mu)
    H, g, Sc, c0, idx = condensed_qp(x0, r, stance, xd, delta, feats["w_stage"][b], f["force"], f["torque"],
                                     mass=f["mass"], ibody_inv=f["ibody_inv"], r_weight=f["r_weight"])
    legs = co.stance_legs(idx, f["normal"], f["mu"], f["f_min"], f["f_max"])
    if "f_ref" in feats:
        H, g = fo.add_force_ref(H, g, idx, feats["f_ref"][b], feats["f_weight"][b])
    return H, g, Sc, c0, idx, legs


def mix_admm(pb, b, feats, delta=DT, as_f32=False, **admm_kw):
    """contact_oracle.admm on problem b's QP with every feature (keywords as condensed_admm.admm)"""
    x0, r, stance, xd, mu = mo.problem(pb, b, as_f32)
    H, g, Sc, c0, idx, legs = mix_qp(pb, b, feats, delta, as_f32)
    return bo._finish(co.admm(H, g, *legs, **admm_kw), r, xd, Sc, c0, idx, H, g)
