"""fp64 statement of a problem with every per-slot feature at once (cmpc_set_body, cmpc_set_contact,
cmpc_set_weights and cmpc_set_wrench on one slot) for the tests: wrench_oracle's QP with the slot's body and
weights, solved by contact_oracle's ADMM with the slot's surfaces, and X with the wrench's free response.

``feats`` holds per-slot arrays over the batch, in the fp32-rounded fp64 the device holds:
    mass (B,), ibody_inv (B,3,3) or (B,3)           - cmpc_set_body
    normal (B,N,4,3), mu, f_min, f_max (B,N,4)      - cmpc_set_contact
    w (B,13), r_weight (B,)                         - cmpc_set_weights
    force, torque (B,N,3)                           - cmpc_set_wrench
A group that is missing takes the configuration's defaults, as a slot that was never set does: the default body,
flat ground with the call's mu and the configured f_min / f_max, the default weights and no wrench.  Each single
group reduces this to the oracle of that feature (tests/test_mix_oracle_cpu.py checks it).
"""
import numpy as np

from oracle import srbd_qp
from mpc_b200.problems import DT
import body_oracle as bo
import contact_oracle as co
import wrench_oracle as wo


def r32(a):
    """what the device holds, in fp64 for the oracle"""
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def problem(pb, b, as_f32=False):
    """(x0, r, stance, x_des (13,N+1), mu) of problem b; as_f32: the fp32 data the kernel reads."""
    x0, r, stance, xd, mu = pb.problem(b)
    if as_f32:
        x0, r, xd, mu = r32(x0), r32(r), r32(xd), float(np.float32(mu))
    return x0, r, stance, xd, mu


def slot_features(feats, b, N, mu):
    """The features of problem b with the defaults filled in: a dict of the keyword arguments of
    wrench_oracle.condensed_qp (mass, ibody_inv, w, r_weight), force, torque and the contacts (N,4,...)."""
    f = dict(mass=srbd_qp.MASS, ibody_inv=srbd_qp.IBODY_INV, w=srbd_qp.W_STATE, r_weight=0.0,
             force=np.zeros((N, 3)), torque=np.zeros((N, 3)), normal=np.tile([0.0, 0.0, 1.0], (N, 4, 1)),
             mu=np.full((N, 4), mu), f_min=np.full((N, 4), srbd_qp.F_MIN), f_max=np.full((N, 4), srbd_qp.F_MAX))
    for k in f:
        if k in feats:
            f[k] = feats[k][b]
    f["r_weight"] = float(f["r_weight"])
    return f


def mix_qp(pb, b, feats, delta=DT, as_f32=False):
    """(H, g, Sc, c0, idx, legs) of problem b under its slot's features; legs = contact_oracle.stance_legs, the
    (R, mu, f_min, f_max) of each stance leg-stage in the order of the QP's unknowns."""
    x0, r, stance, xd, mu = problem(pb, b, as_f32)
    f = slot_features(feats, b, r.shape[0], mu)
    H, g, Sc, c0, idx = wo.condensed_qp(x0, r, stance, xd, delta, f["force"], f["torque"], w=f["w"], mass=f["mass"],
                                        ibody_inv=f["ibody_inv"], r_weight=f["r_weight"])
    legs = co.stance_legs(idx, f["normal"], f["mu"], f["f_min"], f["f_max"])
    return H, g, Sc, c0, idx, legs


def project(x, legs):
    """Projection of the stacked stance forces x onto the product of their rotated frustums."""
    return co.project(np.asarray(x, dtype=float).reshape(-1, 3), *legs).reshape(-1)


def mix_admm(pb, b, feats, delta=DT, as_f32=False, **admm_kw):
    """contact_oracle.admm on problem b's QP (keywords as condensed_admm.admm); U (N,12), X (13,N+1) including the
    wrench's response, and the ADMM's x, y, z."""
    x0, r, stance, xd, mu = problem(pb, b, as_f32)
    H, g, Sc, c0, idx, legs = mix_qp(pb, b, feats, delta, as_f32)
    return bo._finish(co.admm(H, g, *legs, **admm_kw), r, xd, Sc, c0, idx, H, g)
