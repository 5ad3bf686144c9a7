"""The two formulations of the solve kernel - dense single-CTA (default for N <= 16) and stage-wise
Riccati (default for N >= 20), the other one selected by `kernel_variant` = 5: same ADMM, same iterates,
so the same oracle checks apply to both."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import mpc_b200 as pkg                                          # noqa: E402
from mpc_b200.problems import synthetic_batch, DT, GAIT_NAMES     # noqa: E402
from oracle import condensed_admm as ca, srbd_qp                 # noqa: E402
from test_gpu_parity import gpu_solve, close, ATOL, RTOL, _FakeLite3, _Logger   # noqa: E402


@pytest.mark.parametrize("N,variant,gaits", [(40, 0, ("trot",)), (60, 0, ("pseudo_gallop",)), (30, 0, GAIT_NAMES),
                                             (20, 0, GAIT_NAMES), (30, 0, ("trot",)),
                                             # variant 5 = the other formulation: stage-wise (Riccati) kernel
                                             # for N <= 16 (default: dense), dense kernel for N = 20 / 30
                                             # (default: Riccati)
                                             (10, 5, GAIT_NAMES), (12, 5, GAIT_NAMES), (16, 5, GAIT_NAMES),
                                             (20, 5, GAIT_NAMES), (30, 5, GAIT_NAMES)])
def test_cluster_kernel_iterate_parity(N, variant, gaits):
    assert pkg._capi.has_variant(N, variant)
    B, K = 6, (50 if N < 60 else 120)
    pb = synthetic_batch(B, N=N, gaits=gaits, seed=3)
    out = gpu_solve(pb, max_iter=K, check_every=100000, eps_abs=0.0, eps_rel=0.0, warm_mode=0,
                    adaptive_rho_interval=0, kernel_variant=variant)
    assert np.all(out["iters"] == K)
    for b in range(B):
        x0, r, stance, xd, mu = pb.problem(b)
        ref = ca.solve_problem(x0, r, stance, xd, mu, DT, fixed_iters=K, rho=float(out["mpc"].cfg.rho))
        err = np.abs(out["U"][b] - ref["U"])
        # transient comparison: the fp32 Woodbury step error grows with the horizon (kappa ~ N^2)
        tr = (3e-3 if N < 60 else 6e-3) * np.abs(ref["U"]).max()
        assert np.all(err <= 2 * ATOL + tr + RTOL * np.abs(ref["U"])), (b, err.max())
        assert close(out["X"][b].T, ref["X"], atol=2e-4, rtol=1e-3)
        sw = np.repeat(pb.stance[b].reshape(-1) == 0, 3)
        assert np.all(out["U"][b].reshape(-1)[sw] == 0.0)


@pytest.mark.parametrize("N,variant", [(60, 0), (30, 5)])
def test_cluster_kernel_converges_like_the_single_cta_kernel(N, variant):
    pb = synthetic_batch(24, N=N, seed=12)
    a = gpu_solve(pb, kernel_variant=variant)
    assert np.mean(a["status"] == 1) >= 0.9
    for b in range(0, 24, 6):
        if a["status"][b] != 1:
            continue
        x0, r, stance, xd, mu = pb.problem(b)
        tight = ca.solve_problem(x0, r, stance, xd, mu, DT, tight=True, rho=0.3, max_iter=20000,
                                 eps_abs=1e-7, eps_rel=1e-7)
        J = srbd_qp.objective(a["X"][b].T, xd)
        assert abs(J / tight["J"] - 1.0) < 2e-2
    if N == 30:          # same problems through the default (Riccati) kernel: same iterations, same forces
        s = gpu_solve(pb, kernel_variant=0)
        assert np.array_equal(s["status"], a["status"])
        assert np.abs(s["iters"].astype(int) - a["iters"].astype(int)).max() <= 10


def test_dropin_at_the_reference_default_horizon(gold):
    """The reference's own configuration (N = 60, src/main.py:41): the drop-in MPC on the
    golden run's states; objective within 2 % of the tight fp64 optimum of every tick."""
    from oracle.replay import params_from_golden, initial_from_golden, ReplayMPC
    params = params_from_golden(gold)          # N = 60
    initial = initial_from_golden(gold)
    gp = pkg.GaitPlan.from_initial(initial, params)
    lite3, logger = _FakeLite3(gold), _Logger()
    mpc = pkg.MPC(lite3=lite3, initial=initial_from_golden(gold), footstep_planner=gp, params=params)
    rep = ReplayMPC(initial_from_golden(gold), params)
    for t in range(6):
        lite3.t = t
        forces = mpc.solve(t, logger)
        assert mpc.x_log.shape == (12, 61) and mpc.u_plot.shape == (12, 60)
        assert np.array_equal(logger.track[-1][1], gold["desired"][t])
        x0, r, stance, xd, v, om = rep.tick_problem(t, gold["state"][t], gold["feet"][t])
        rep.com_pos_start = rep.com_pos_start + v * 0.01
        rep.yaw_start = rep.yaw_start + om * 0.01
        if t in (0, 5):
            tight = ca.solve_problem(x0, r, stance, xd, 1.0, 0.01, tight=True, eps_abs=1e-6, eps_rel=1e-6,
                                     max_iter=20000)
            J = srbd_qp.objective(np.vstack([mpc.x_log, np.full((1, 61), params["g"])]), xd)
            assert abs(J / tight["J"] - 1.0) < 2e-2, (t, J, tight["J"])
        fz = sum(forces[leg][2] for leg in pkg.LEGS)
        assert 40.0 < fz < 200.0
