"""fp64 restatement of per-foot contact surfaces (cmpc_set_contact) for the tests: the QP of one problem with each
stance leg-stage's force kept in the friction frustum of its own surface, R_l C(mu_l, f_min_l, f_max_l), where
R_l = [t1 t2 n] is the contact frame of the leg-stage's normal.

The oracle package models flat ground with one mu and the configuration's bounds, and stays as it is.  The
functions here follow ``oracle.condensed_admm.admm`` and ``oracle.tight_ipm.solve_qp`` line for line with per-leg
frames, mu and bounds, so that flat normals with the problem's mu and the default bounds reproduce the oracle's
numbers exactly (``tests/test_contact_cpu.py`` checks that).  The QP comes from ``body_oracle.condensed_qp``, so
bodies and contacts compose.
"""
import numpy as np
import scipy.linalg as sla

from oracle import condensed_admm as ca, srbd_qp, tight_ipm as ipm
import body_oracle as bo


def contact_frame(normal):
    """(...,3) -> R (...,3,3) with columns t1, t2, n:  n = normal/|normal|; t1 = normalise(e_x - n_x n) if
    n_x^2 <= 1/2, else normalise(e_y - n_y n); t2 = n x t1."""
    normal = np.asarray(normal, dtype=float)
    n = normal / np.linalg.norm(normal, axis=-1, keepdims=True)
    use_x = n[..., 0] ** 2 <= 0.5
    e = np.where(use_x[..., None], np.array([1.0, 0.0, 0.0]), np.array([0.0, 1.0, 0.0]))
    v = e - np.where(use_x, n[..., 0], n[..., 1])[..., None] * n
    t1 = v / np.linalg.norm(v, axis=-1, keepdims=True)
    t2 = np.cross(n, t1)
    return np.stack([t1, t2, n], axis=-1)


def project(w, R, mu, f_min=srbd_qp.F_MIN, f_max=srbd_qp.F_MAX):
    """Euclidean projection of w (...,3) onto the rotated frustum R C(mu, f_min, f_max):  R P_C(R' w)."""
    local = np.einsum("...ji,...j->...i", R, w)
    return np.einsum("...ij,...j->...i", R, ca.project_frustum(local, mu, f_min, f_max))


def stance_legs(idx, normal, mu, f_min, f_max):
    """Per stance leg-stage (in the order of srbd_qp.stance_index) of (N,4,...) contacts: R, mu, f_min, f_max."""
    sel = tuple(np.array([ij[k] for ij in idx], dtype=int) for k in (0, 1))
    R = contact_frame(np.asarray(normal, dtype=float)[sel])
    return R, np.asarray(mu, dtype=float)[sel], np.asarray(f_min, dtype=float)[sel], np.asarray(f_max, dtype=float)[sel]


def admm(H, g, R, mu, f_min, f_max, rho=0.3, sigma=1e-6, alpha=1.6, eps_abs=1e-3, eps_rel=1e-3,
         max_iter=1000, check_every=5, x=None, y=None, dtype=np.float64, fixed_iters=None, adaptive_interval=0,
         adaptive_tolerance=2.0, rho_lim=(0.03, 30.0), adaptive_floor=0.0):
    """condensed_admm.admm with the projection of each stance leg onto its own rotated frustum (R, mu, f_min,
    f_max per stance leg)."""
    n = H.shape[0]
    dt = dtype
    H = H.astype(dt)
    g = g.astype(dt)
    x = np.zeros(n, dt) if x is None else x.astype(dt)
    y = np.zeros(n, dt) if y is None else y.astype(dt)
    proj = lambda v: project(v.reshape(-1, 3), R, mu, f_min, f_max).reshape(-1).astype(dt)
    z = proj(x)
    rho, sigma, alpha = dt(rho), dt(sigma), dt(alpha)

    def factor(rho_):
        K = H + (sigma + rho_) * np.eye(n, dtype=dt)
        return np.linalg.cholesky(K.astype(np.float64)).astype(dt) if dt == np.float64 \
            else ca._chol32(K)
    if n:
        L = factor(rho)
    rho_updates = 0
    status, it = 0, 0
    pri = dua = dt(0)
    total = fixed_iters if fixed_iters is not None else max_iter

    def residuals():
        Hx = H @ x
        pri_ = ca._inf(x - z)
        dua_ = ca._inf(Hx + g + y)
        return pri_, dua_, max(ca._inf(x), ca._inf(z)), max(ca._inf(Hx), ca._inf(y), ca._inf(g))

    if fixed_iters is None and n == 0:
        return dict(x=x, y=y, z=z, iters=0, pri_res=0.0, dua_res=0.0, status=1, rho=float(rho),
                    rho_updates=0)
    if fixed_iters is None:
        pri, dua, nA, nD = residuals()
        if pri <= eps_abs + eps_rel * nA and dua <= eps_abs + eps_rel * nD:
            return dict(x=x, y=y, z=z, iters=0, pri_res=pri, dua_res=dua, status=1,
                        rho=float(rho), rho_updates=0)
    for it in range(1, total + 1):
        rhs = sigma * x - g + rho * z - y
        xt = ca._chol_solve(L, rhs) if n else rhs
        x = alpha * xt + (1 - alpha) * x
        zh = alpha * xt + (1 - alpha) * z
        zn = proj(zh + y / rho)
        y = y + rho * (zh - zn)
        z = zn
        adapt = adaptive_interval > 0 and it % adaptive_interval == 0
        if (fixed_iters is None and it % check_every == 0) or adapt:
            pri, dua, nA, nD = residuals()
            if fixed_iters is None and pri <= eps_abs + eps_rel * nA and dua <= eps_abs + eps_rel * nD:
                status = 1
                break
            if adapt and n and max(pri / (nA + 1e-10), dua / (nD + 1e-10)) > adaptive_floor:
                rn = float(rho) * np.sqrt((pri / (nA + 1e-10)) / (dua / (nD + 1e-10) + 1e-10))
                rn = min(max(rn, rho_lim[0]), rho_lim[1])
                if rn > float(rho) * adaptive_tolerance or rn * adaptive_tolerance < float(rho):
                    rho = dt(rn)
                    L = factor(rho)
                    rho_updates += 1
    if fixed_iters is not None or status == 0:
        pri, dua, _, _ = residuals()
    return dict(x=x, y=y, z=z, iters=it, pri_res=float(pri), dua_res=float(dua), status=status,
                rho=float(rho), rho_updates=rho_updates)


def leg_rows(R, mu, f_min, f_max):
    """C (6,3), d (6,) of one stance leg on its surface:  C1(mu) R' f <= d."""
    C1, d = ipm.leg_rows(mu, f_min, f_max)
    return C1 @ R.T, d


def solve_qp(H, g, R, mu, f_min, f_max, tol=1e-11, max_iter=100):
    """tight_ipm.solve_qp with per-leg rows C1(mu_l) R_l' f <= d(f_min_l, f_max_l).  Legs with the same rows are
    handled together, with the oracle's operations (one group for flat ground with one mu)."""
    n = H.shape[0]
    if n == 0:
        return dict(x=np.zeros(0), lam=np.zeros(0), iters=0, gap=0.0, res=0.0)
    nl = n // 3
    rows = [leg_rows(R[l], mu[l], f_min[l], f_max[l]) for l in range(nl)]
    groups = {}
    for l, (C_l, d_l) in enumerate(rows):
        groups.setdefault((C_l.tobytes(), d_l.tobytes()), []).append(l)
    groups = [(rows[ls[0]][0], np.array(ls)) for ls in groups.values()]
    d = np.concatenate([d_l for (_, d_l) in rows])

    def Cmul(x):                     # (6 nl,)
        out = np.empty((nl, 6))
        X = x.reshape(nl, 3)
        for C1, ls in groups:
            out[ls] = X[ls] @ C1.T
        return out.reshape(-1)

    def Ctmul(v):                    # (n,)
        out = np.empty((nl, 3))
        V = v.reshape(nl, 6)
        for C1, ls in groups:
            out[ls] = V[ls] @ C1
        return out.reshape(-1)

    # strictly feasible start: f.n at the middle of its range, no tangential force
    x = np.concatenate([R[l] @ np.array([0.0, 0.0, 0.5 * (f_min[l] + f_max[l])]) for l in range(nl)])
    s = d - Cmul(x)
    scale = max(1.0, float(np.abs(g).max()), float(np.abs(H).max()))
    lam = np.full(6 * nl, 1.0) * max(1.0, scale * 1e-3)
    it = 0
    for it in range(1, max_iter + 1):
        rd = H @ x + g + Ctmul(lam)                  # dual residual
        rp = Cmul(x) + s - d                         # primal residual (0 after a full step)
        mu_c = float(s @ lam) / (6 * nl)
        if max(np.abs(rd).max() / scale, np.abs(rp).max(), mu_c / scale) < tol:
            break
        w = lam / s
        blocks = np.empty((nl, 3, 3))
        for C1, ls in groups:
            blocks[ls] = np.einsum("ki,lk,kj->lij", C1, w.reshape(nl, 6)[ls], C1)
        Kmat = H.copy()
        for l in range(nl):
            Kmat[3 * l:3 * l + 3, 3 * l:3 * l + 3] += blocks[l]
        reg = 1e-13 * scale
        while True:
            try:
                cf = sla.cho_factor(Kmat + reg * np.eye(n), lower=True, check_finite=False)
                break
            except np.linalg.LinAlgError:
                reg *= 100.0

        def newton(rc):
            rhs = -rd - Ctmul((rc - lam * rp) / s * -1.0)
            dx = sla.cho_solve(cf, rhs, check_finite=False)
            ds = -rp - Cmul(dx)
            dl = -(rc + lam * ds) / s
            return dx, ds, dl

        dx, ds, dl = newton(s * lam)                 # affine (predictor)
        a_p = ipm._step(s, ds)
        a_d = ipm._step(lam, dl)
        mu_aff = float((s + a_p * ds) @ (lam + a_d * dl)) / (6 * nl)
        sig = (mu_aff / mu_c) ** 3 if mu_c > 0 else 0.0
        dx, ds, dl = newton(s * lam + ds * dl - sig * mu_c)   # corrector
        a_p = min(1.0, 0.995 * ipm._step(s, ds))
        a_d = min(1.0, 0.995 * ipm._step(lam, dl))
        x = x + a_p * dx
        s = s + a_p * ds
        lam = lam + a_d * dl
    return dict(x=x, lam=lam, iters=it, gap=float(s @ lam) / (6 * nl),
                res=float(np.abs(H @ x + g + Ctmul(lam)).max()))


def admm_solve(x0, r, stance, x_des, delta, normal, mu, f_min, f_max, mass=srbd_qp.MASS,
               ibody_inv=srbd_qp.IBODY_INV, **kw):
    """condensed_admm.solve_problem (r_weight = 0) for the given contacts (N,4,3) / (N,4) and body."""
    H, gvec, Sc, c0, idx = bo.condensed_qp(x0, r, stance, x_des, delta, mass=mass, ibody_inv=ibody_inv)
    info = admm(H, gvec, *stance_legs(idx, normal, mu, f_min, f_max), **kw)
    return bo._finish(info, r, x_des, Sc, c0, idx, H, gvec)


def ipm_solve(x0, r, stance, x_des, delta, normal, mu, f_min, f_max, mass=srbd_qp.MASS,
              ibody_inv=srbd_qp.IBODY_INV, **kw):
    """tight_ipm.solve_problem (r_weight = 0) for the given contacts (N,4,3) / (N,4) and body."""
    H, gvec, Sc, c0, idx = bo.condensed_qp(x0, r, stance, x_des, delta, mass=mass, ibody_inv=ibody_inv)
    info = solve_qp(H, gvec, *stance_legs(idx, normal, mu, f_min, f_max), **kw)
    return bo._finish(info, r, x_des, Sc, c0, idx, H, gvec)
