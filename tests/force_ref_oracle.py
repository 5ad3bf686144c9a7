"""fp64 statement of the per-robot force references (cmpc_set_force_ref) for the tests: the objective gains
sum over stance leg-stages (i, l) of w_f[i,l] ||f[i,l] - f_ref[i,l]||^2, which in condensed form is
H += 2 w_f I and g -= 2 w_f f_ref on the three unknowns of each stance pair of ``idx``.  Swing leg-stages have no
unknowns and ignore their entries.  The functions wrap body_oracle.condensed_qp and mix_oracle.mix_qp unchanged.

``feats`` (mix_qp, mix_admm) is mix_oracle's dict with two more per-slot arrays: f_ref (B,N,4,3) and f_weight
(B,N,4); without them the problem has no reference.
"""
import numpy as np

from mpc_b200.problems import DT
import body_oracle as bo
import contact_oracle as co
import mix_oracle as mo


def add_force_ref(H, g, idx, f_ref, weight):
    """(H + 2 diag(w_f), g - 2 w_f f_ref) over the stance pairs idx; f_ref (N,4,3), weight (N,4)"""
    H, g = H.copy(), g.copy()
    for s, (i, l) in enumerate(idx):
        w = float(weight[i, l])
        H[3 * s:3 * s + 3, 3 * s:3 * s + 3] += 2.0 * w * np.eye(3)
        g[3 * s:3 * s + 3] -= 2.0 * w * np.asarray(f_ref[i, l], dtype=float)
    return H, g


def condensed_qp(x0, r, stance, x_des, delta, f_ref, weight, **kw):
    """body_oracle.condensed_qp (keywords: w, mass, ibody_inv, r_weight) with the force reference: (H, g, Sc, c0, idx)"""
    H, g, Sc, c0, idx = bo.condensed_qp(x0, r, stance, x_des, delta, **kw)
    H, g = add_force_ref(H, g, idx, f_ref, weight)
    return H, g, Sc, c0, idx


def mix_qp(pb, b, feats, delta=DT, as_f32=False):
    """mix_oracle.mix_qp with the slot's force reference: (H, g, Sc, c0, idx, legs)"""
    H, g, Sc, c0, idx, legs = mo.mix_qp(pb, b, feats, delta, as_f32)
    if "f_ref" in feats:
        H, g = add_force_ref(H, g, idx, feats["f_ref"][b], feats["f_weight"][b])
    return H, g, Sc, c0, idx, legs


def mix_admm(pb, b, feats, delta=DT, as_f32=False, **admm_kw):
    """contact_oracle.admm on problem b's QP with every feature (keywords as condensed_admm.admm)"""
    x0, r, stance, xd, mu = mo.problem(pb, b, as_f32)
    H, g, Sc, c0, idx, legs = mix_qp(pb, b, feats, delta, as_f32)
    return bo._finish(co.admm(H, g, *legs, **admm_kw), r, xd, Sc, c0, idx, H, g)
