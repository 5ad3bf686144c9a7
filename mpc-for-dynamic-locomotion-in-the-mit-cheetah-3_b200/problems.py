"""Batched gait plans and synthetic MPC workloads (numpy, fp64, vectorised over robots).

``BatchedGaitPlan`` is the array-of-robots form of :class:`gait.GaitPlan`: every robot
may have its own gait (first_swing, ss, ds), reference velocity and yaw rate, so the
unicycle integration of reference ``src/footstep_planner.py:72-177`` is carried out for
all robots at once.  ``synthetic_batch`` draws the workloads SURVEY.md section 8(d)
defines for BASELINE.json's configs 2-4 (randomised CoM states / velocity references
around a walking Lite3) and assembles the per-problem QP parameters exactly as the
reference's ``MPC.solve`` would (``src/mpc.py:178-255``).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from .gait import GAITS, stance_bits

# pkl tick 0 of the reference's logged run (SURVEY.md section 8d)
NOMINAL_FEET = np.array([[0.10629492, 0.1605, 0.01713467],
                         [0.10629492, -0.1605, 0.01713467],
                         [-0.24270508, 0.1605, 0.01713467],
                         [-0.24270508, -0.1605, 0.01713467]])
NOMINAL_COM = np.array([-0.0101835626879727, -0.00027996234635044087, 0.285])
GRAVITY = -9.81
DT = 0.01
_SGN_T = np.array([+1.0, +1.0, -1.0, -1.0])    # torso_displacement/2 sign, FL FR HL HR
_SGN_L = np.array([-1.0, +1.0, -1.0, +1.0])    # leg_displacement_y sign


@dataclass
class BatchedGaitPlan:
    pos: np.ndarray        # (B,S,4,3)
    feet_id: np.ndarray    # (B,S,4) stance mask of each step's single-support part
    ss: np.ndarray         # (B,) int
    ds: np.ndarray         # (B,) int
    step_height: float = 0.08

    @classmethod
    def build(cls, feet0, yaw0, first_swing, ss, ds, v_ref, omega_ref, total_steps=20,
              dt=DT, step_height=0.08) -> "BatchedGaitPlan":
        """feet0 (B,4,3) or (4,3); yaw0 (B,); first_swing (B,4); ss, ds (B,) ints;
        v_ref (B,3); omega_ref (B,)."""
        first_swing = np.atleast_2d(np.asarray(first_swing)).astype(np.int64)
        B = first_swing.shape[0]
        feet0 = np.broadcast_to(np.asarray(feet0, dtype=float), (B, 4, 3))
        ss = np.broadcast_to(np.asarray(ss, dtype=np.int64), (B,)).copy()
        ds = np.broadcast_to(np.asarray(ds, dtype=np.int64), (B,)).copy()
        v_ref = np.broadcast_to(np.asarray(v_ref, dtype=float), (B, 3))
        omega_ref = np.broadcast_to(np.asarray(omega_ref, dtype=float), (B,))
        theta = np.broadcast_to(np.asarray(yaw0, dtype=float), (B,)).copy()
        S = int(total_steps)
        # same arithmetic, in the same order, as reference src/footstep_planner.py:72-177 (and
        # gait.GaitPlan.from_initial): the 2x2 rotations go through np.matmul like the reference's
        # `Rm @ v`, so that the plan of every robot agrees with the reference planner to the last bit
        fl, fr, hl, hr = feet0[:, 0], feet0[:, 1], feet0[:, 2], feet0[:, 3]
        uni = (hl + hr + fl + fr) / 4.0                   # (B,3)
        dfl = fl[:, :2] - hl[:, :2]
        dlat = hr[:, :2] - hl[:, :2]

        def rot(th):
            c, s = np.cos(th), np.sin(th)
            return np.stack([np.stack([c, -s], -1), np.stack([s, c], -1)], -2)      # (B,2,2)

        def apply(Rm, v):                                  # per-robot Rm @ v (stacked matmul: same BLAS
            return np.matmul(Rm, v[:, :, None])[:, :, 0]   # kernel, same bits as the reference's 2x2 `@`)

        pos = np.zeros((B, S, 4, 3))
        feet_id = np.ones((B, S, 4), dtype=np.int64)
        support = first_swing.copy()
        period = ss + ds
        Rm = rot(theta)
        for j in range(S):
            if j >= 1:
                for i in range(int(period.max())):
                    live = i < period
                    theta = np.where(live, theta + omega_ref * dt, theta)
                    Rm = np.where(live[:, None, None], rot(theta), Rm)
                    step = apply(Rm, v_ref[:, :2]) * dt
                    uni[:, :2] = np.where(live[:, None], uni[:, :2] + step, uni[:, :2])
            torso = apply(Rm, dfl)
            lat = apply(Rm, dlat) / 2.0
            half = torso / 2
            base = uni[:, None, :2] + _SGN_T[None, :, None] * half[:, None, :]     # u +- t/2 (exact sign flip)
            new = np.empty((B, 4, 3))
            new[:, :, :2] = base + _SGN_L[None, :, None] * lat[:, None, :]          # (u +- t/2) +- lat
            new[:, :, 2] = uni[:, None, 2]
            if j >= 1:
                keep = support.astype(bool)[:, :, None]
                pos[:, j] = np.where(keep, pos[:, j - 1], new)
                feet_id[:, j] = support
                support = 1 - support
            else:
                pos[:, j] = new
        return cls(pos, feet_id, ss, ds, step_height)

    @property
    def n_steps(self):
        return self.pos.shape[1]

    def step_index(self, t):
        """t (B,) or (B,K) ticks -> step index, reference src/footstep_planner.py:226-231."""
        t = np.asarray(t)
        period = (self.ss + self.ds).reshape((-1,) + (1,) * (t.ndim - 1))
        return np.minimum(t // period, self.n_steps - 1)

    def stance_mask(self, t):
        """(B,K) ticks -> (B,K,4) stance mask, reference src/footstep_planner.py:239-246."""
        t = np.asarray(t)
        shp = (-1,) + (1,) * (t.ndim - 1)
        step = self.step_index(t)
        tin = t - step * (self.ss + self.ds).reshape(shp)
        single = tin < self.ss.reshape(shp)
        b = np.arange(t.shape[0]).reshape(shp)
        return np.where(single[..., None], self.feet_id[b, step], 1)

    def foot_position(self, t):
        """(B,K) ticks -> (B,K,4,3) look-ahead foot position (reference src/mpc.py:306-318,
        src/foot_trajectory_generator.py:27-96)."""
        t = np.asarray(t)
        shp = (-1,) + (1,) * (t.ndim - 1)
        step = self.step_index(t)
        b = np.arange(t.shape[0]).reshape(shp)
        tin = (t - step * (self.ss + self.ds).reshape(shp)).astype(float)[..., None, None]
        start = self.pos[b, step]
        target = self.pos[b, np.minimum(step + 1, self.n_steps - 1)]
        ts = (0.80 * self.ss.astype(float)).reshape(shp)[..., None, None]
        out = start + (target - start) * (-2 / ts ** 3 * tin ** 3 + 3 / ts ** 2 * tin ** 2)
        h = self.step_height
        tz, tsz = tin[..., 0], ts[..., 0]
        out[..., 2] = (16 * h / tsz ** 4 * tz ** 4 - 32 * h / tsz ** 3 * tz ** 3
                       + 16 * h / tsz ** 2 * tz ** 2 + start[..., 2])
        out = np.where(tin >= ts, target, out)
        out = np.where((step == 0)[..., None, None], start, out)
        stance = self.stance_mask(t).astype(bool)[..., None]
        return np.where(stance, start, out)


@dataclass
class ProblemBatch:
    """fp64 problem data in the layout of the C ABI (SURVEY.md section 8b)."""
    x0: np.ndarray        # (B,13)
    r: np.ndarray         # (B,N,4,3)
    stance: np.ndarray    # (B,N,4) {0,1}
    x_des: np.ndarray     # (B,N+1,13)
    mu: np.ndarray        # (B,)
    gait_id: np.ndarray   # (B,)
    tick: np.ndarray      # (B,)

    @property
    def B(self):
        return self.x0.shape[0]

    @property
    def N(self):
        return self.r.shape[1]

    @property
    def mask_bits(self):
        return stance_bits(self.stance)

    def f32(self):
        """(x0, r, mask, x_des, mu) as contiguous fp32/uint8 numpy arrays."""
        c = np.ascontiguousarray
        return (c(self.x0, dtype=np.float32), c(self.r, dtype=np.float32), c(self.mask_bits),
                c(self.x_des, dtype=np.float32), c(self.mu, dtype=np.float32))

    def problem(self, b):
        """(x0, r, stance, x_des(13,N+1), mu) of problem b for the oracle."""
        return self.x0[b], self.r[b], self.stance[b], self.x_des[b].T, float(self.mu[b])

    def slice(self, lo, hi):
        return ProblemBatch(self.x0[lo:hi], self.r[lo:hi], self.stance[lo:hi], self.x_des[lo:hi],
                            self.mu[lo:hi], self.gait_id[lo:hi], self.tick[lo:hi])


GAIT_NAMES = ("trot", "pronk", "amble", "pseudo_gallop")


def synthetic_batch(B, N=10, gaits=("trot",), seed=0, mu=(1.0, 1.0), tick_range=(20, 380),
                    noise=1.0, total_steps=20, tick_shift=0) -> ProblemBatch:
    """Workload of BASELINE.json configs 2-4 (SURVEY.md section 8d): robot b walks with gait
    ``gaits[b % len(gaits)]``... drawn uniformly; tick ~ U{tick_range}; velocity references
    v_x ~ U[-0.3,0.3], v_y ~ U[-0.1,0.1], yaw rate ~ U[-0.5,0.5]; measured state = reference
    state at that tick + N(0, sigma) noise (rpy 0.05 rad, com 0.02 m, omega 0.2 rad/s,
    v 0.1 m/s); stage-0 feet = planned feet + N(0, 0.005 m); mu ~ U[mu].
    ``tick_shift`` moves every robot's tick by that many ticks with all random draws unchanged
    (``tick_shift=-1`` is "the same problems one tick earlier", the warm-start source of config 2)."""
    rng = np.random.default_rng(seed)
    gid = rng.integers(0, len(gaits), size=B)
    table = [GAITS[g] for g in gaits]
    first_swing = np.array([table[i][0] for i in gid], dtype=np.int64)
    ss = np.array([table[i][1] for i in gid], dtype=np.int64)
    ds = np.array([table[i][2] for i in gid], dtype=np.int64)
    tick = rng.integers(tick_range[0], tick_range[1], size=B) + int(tick_shift)
    v_ref = np.stack([rng.uniform(-0.3, 0.3, B), rng.uniform(-0.1, 0.1, B), np.zeros(B)], 1)
    om_ref = rng.uniform(-0.5, 0.5, B)
    mu_b = rng.uniform(mu[0], mu[1], B)
    plan = BatchedGaitPlan.build(NOMINAL_FEET, np.zeros(B), first_swing, ss, ds, v_ref, om_ref,
                                 total_steps=total_steps)
    # reference (src/mpc.py:181-183): references are zeroed during the last planned step
    last = plan.step_index(tick) == total_steps - 1
    v_use = np.where(last[:, None], 0.0, v_ref)
    om_use = np.where(last, 0.0, om_ref)
    # reference accumulators after `tick` solves (src/mpc.py:261-262), all before the last step
    yaw_start = om_ref * DT * tick
    com_start = NOMINAL_COM[None] + v_ref * DT * tick[:, None]
    k = np.arange(N + 1)
    x_des = np.zeros((B, N + 1, 13))
    x_des[:, :, 2] = yaw_start[:, None] + om_use[:, None] * DT * k
    x_des[:, :, 3:6] = com_start[:, None, :] + v_use[:, None, :] * DT * k[None, :, None]
    x_des[:, :, 8] = om_use[:, None]
    x_des[:, :, 9:12] = v_use[:, None, :]
    x_des[:, :, 12] = GRAVITY
    x0 = x_des[:, 0, :].copy()
    x0[:, 0:3] += noise * rng.normal(0, 0.05, (B, 3))
    x0[:, 3:6] += noise * rng.normal(0, 0.02, (B, 3))
    x0[:, 6:9] += noise * rng.normal(0, 0.2, (B, 3))
    x0[:, 9:12] += noise * rng.normal(0, 0.1, (B, 3))
    ticks = tick[:, None] + np.arange(N)[None]
    feet = plan.foot_position(ticks)                                   # (B,N,4,3)
    feet[:, 0] += noise * rng.normal(0, 0.005, (B, 4, 3))
    r = np.empty((B, N, 4, 3))
    r[:, 0] = feet[:, 0] - x0[:, None, 3:6]                            # measured (src/mpc.py:223-226)
    r[:, 1:] = feet[:, 1:] - x_des[:, 1:N, None, 3:6]                  # planned - desired com
    stance = plan.stance_mask(ticks)
    return ProblemBatch(x0, r, stance, x_des, mu_b, gid, tick)


# reference body (src/mpc.py:71-76): principal inertias of the Lite3 torso, kg m^2
REF_MASS = 8.885
REF_INERTIA = np.array([0.24, 1.0, 1.0])


def random_bodies(B, seed=0, mass_range=(0.75, 1.35), inertia_range=(0.7, 1.4), max_tilt=0.15):
    """Per-robot rigid bodies for domain randomisation / payload sweeps (fp64):
    mass (B,) = U(mass_range) x the reference's 8.885 kg, and the body-frame inverse inertia
    ibody_inv (B,3,3) = R diag(1/I) R' with principal inertias I = U(inertia_range) x the reference's
    and principal axes tilted by a random rotation R of at most `max_tilt` rad, so that it has
    products of inertia.  Draws from its own generator (other draws of the same seed are unaffected)."""
    rng = np.random.Generator(np.random.PCG64(np.random.SeedSequence([int(seed), 0xB0D1])))
    mass = REF_MASS * rng.uniform(*mass_range, size=B)
    inertia = REF_INERTIA * rng.uniform(*inertia_range, size=(B, 3))
    axis = rng.normal(size=(B, 3))
    axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    ang = rng.uniform(0.0, max_tilt, size=B)
    K = np.zeros((B, 3, 3))
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 2] = -axis[:, 2], axis[:, 1], -axis[:, 0]
    K[:, 1, 0], K[:, 2, 0], K[:, 2, 1] = axis[:, 2], -axis[:, 1], axis[:, 0]
    s, c = np.sin(ang)[:, None, None], np.cos(ang)[:, None, None]
    R = np.eye(3) + s * K + (1.0 - c) * (K @ K)            # Rodrigues
    ibody_inv = R @ (np.eye(3) / inertia[:, None, :]) @ np.transpose(R, (0, 2, 1))
    return mass, 0.5 * (ibody_inv + np.transpose(ibody_inv, (0, 2, 1)))


def random_contacts(B, N, seed=0, max_incline_deg=20.0, jitter_deg=3.0, mu_range=(0.3, 1.0), f_min=3.0,
                    f_max_range=(40.0, 100.0)):
    """Per-foot contact surfaces for terrain randomisation (fp64), the arguments of BatchedMPC.set_contact:
    normal (B,N,4,3) = a per-problem incline of up to `max_incline_deg` in a random direction, jittered per
    leg-stage by about `jitter_deg` (unit length); mu (B,N,4) ~ U(mu_range) per leg-stage; f_min (B,N,4) = f_min;
    f_max (B,N,4) ~ U(f_max_range) per leg, the same at every stage.  Draws from its own generator (other draws of
    the same seed are unaffected)."""
    rng = np.random.Generator(np.random.PCG64(np.random.SeedSequence([int(seed), 0xC0A7])))
    tilt = np.radians(max_incline_deg) * rng.uniform(0.0, 1.0, B)
    azim = rng.uniform(0.0, 2.0 * np.pi, B)
    n = np.stack([np.sin(tilt) * np.cos(azim), np.sin(tilt) * np.sin(azim), np.cos(tilt)], 1)
    normal = n[:, None, None, :] + np.radians(jitter_deg) * rng.normal(size=(B, N, 4, 3))
    normal /= np.linalg.norm(normal, axis=-1, keepdims=True)
    mu = rng.uniform(mu_range[0], mu_range[1], (B, N, 4))
    f_max = np.repeat(rng.uniform(f_max_range[0], f_max_range[1], (B, 1, 4)), N, axis=1)
    return normal, mu, np.full((B, N, 4), float(f_min)), f_max


# reference cost weights (src/mpc.py:121-134): Theta, p, omega, v, gravity state
REF_WEIGHTS = np.array([1e4, 2.7e4, 1e4, 2.7e5, 2.7e5, 2.7e5, 1e4, 1e4, 1e4, 1.6e4, 1.6e4, 1.6e4, 0.0])


def random_weights(B, seed=0, spread=4.0):
    """Per-robot cost weights for gain randomisation / weight sweeps (fp64), the arguments of
    BatchedMPC.set_weights: w (B,13) = the reference weights times a log-uniform factor in [1/spread, spread] per
    entry of w[0:12], with w[7] = w[6] (the solver needs equal x/y angular-velocity weights) and w[12] = 0;
    r_weight (B,) = 0 for even b and log-uniform in [1e-5, 1e-2] for odd b.  Draws from its own generator (other
    draws of the same seed are unaffected)."""
    rng = np.random.Generator(np.random.PCG64(np.random.SeedSequence([int(seed), 0x3E16])))
    w = REF_WEIGHTS * np.exp(rng.uniform(-np.log(spread), np.log(spread), (B, 13)))
    w[:, 7] = w[:, 6]
    w[:, 12] = 0.0
    r_weight = np.exp(rng.uniform(np.log(1e-5), np.log(1e-2), B))
    r_weight[0::2] = 0.0
    return w, r_weight


def random_stage_weights(B, N, seed=0):
    """Per-robot stage weights (fp64), the w argument of BatchedMPC.set_stage_weights: w (B,N,13), row i weighing the
    predicted state i + 1, built on the reference weights with w[7] = w[6] and w[12] = 0 on every stage.  Robots cycle
    through four kinds (b mod 4):
      0: one row for the whole horizon, each entry of w[0:12] times a log-uniform factor in [1/4, 4];
      1: a terminal weight: the last stage times a log-uniform factor in [1, 30];
      2: a linear ramp of the whole row from 0.25x to 1x over the horizon, rising or falling (alternately);
      3: a window of stages (never the last) with zero position-like weights w[0:6].
    Every stage keeps positive velocity-like weights, so every robot's weights are valid.  Draws from its own
    generator (other draws of the same seed are unaffected)."""
    rng = np.random.Generator(np.random.PCG64(np.random.SeedSequence([int(seed), 0x57A6])))
    w = np.broadcast_to(REF_WEIGHTS, (B, N, 13)).copy()
    for b in range(B):
        kind = b % 4
        if kind == 0:
            w[b] *= np.exp(rng.uniform(-np.log(4.0), np.log(4.0), 13))
        elif kind == 1:
            w[b, -1] *= np.exp(rng.uniform(0.0, np.log(30.0)))
        elif kind == 2:
            ramp = np.linspace(0.25, 1.0, N) if (b // 4) % 2 == 0 else np.linspace(1.0, 0.25, N)
            w[b] *= ramp[:, None]
        elif N > 1:
            k0 = int(rng.integers(0, N - 1))
            k1 = int(rng.integers(k0 + 1, N))
            w[b, k0:k1, :6] = 0.0
    w[..., 7] = w[..., 6]
    w[..., 12] = 0.0
    return w


def random_force_refs(B, N, seed=0, w_lo=1e-4, w_hi=1e-2):
    """Force references for policy-style randomisation (fp64), the arguments of BatchedMPC.set_force_ref: f_ref
    (B,N,4,3) and weight (B,N,4), world frame, with m g = the reference's 8.885 kg times 9.81 m/s^2.  Each leg-stage's
    reference is a load split near m g / 2 (a trot's two stance legs) with U(0.8, 1.2) jitter on the vertical part
    and a lateral part of U(-0.1, 0.1) m g per axis; each weight is log-uniform in [w_lo, w_hi] (1/N^2 ... 1/N per
    (N/s)^2 against the state cost's O(1) weights).  Even b draw one reference and weight per leg for the whole
    horizon, odd b one per leg-stage.  The default range moves the optimum measurably and keeps every problem
    solvable: on config 2 the stance forces move by 0.99 N on average and 57 N at most, with a SOLVED rate of 1.0
    (scripts/gpu_force_ref_bench.py, NVIDIA B200).  The state cost's curvature on a force is O(10^2-10^3), so weights
    near 1e3 and above make the forces follow the reference closely.
    Draws from its own generator (other draws of the same seed are unaffected)."""
    rng = np.random.Generator(np.random.PCG64(np.random.SeedSequence([int(seed), 0xF0AC])))
    mg = REF_MASS * abs(GRAVITY)
    f_ref = np.empty((B, N, 4, 3))
    f_ref[..., :2] = rng.uniform(-0.1 * mg, 0.1 * mg, (B, N, 4, 2))
    f_ref[..., 2] = 0.5 * mg * rng.uniform(0.8, 1.2, (B, N, 4))
    weight = np.exp(rng.uniform(np.log(w_lo), np.log(w_hi), (B, N, 4)))
    f_ref[0::2] = f_ref[0::2, :1]
    weight[0::2] = weight[0::2, :1]
    return f_ref, weight


def random_wrenches(B, N, seed=0, max_frac=0.2, max_torque=1.0):
    """Known external wrenches for disturbance randomisation (fp64), the arguments of BatchedMPC.set_wrench: force
    (B,N,3) and torque (B,N,3), world frame, with m g = the reference's 8.885 kg times 9.81 m/s^2.
    Even b: a constant wrench over the horizon, a horizontal force of magnitude U(0, max_frac m g) in a direction
    U(0, 2 pi), a vertical force U(-max_frac m g, max_frac m g) and a torque U(-max_torque, max_torque) N m per axis.
    Odd b: a push, the force drawn the same way, on the stages [j0, j0 + L) with j0 ~ U{0..N-1} and
    L ~ U{1..max(1, N // 2)} (cut at N), zero on the other stages; no torque.
    Draws from its own generator (other draws of the same seed are unaffected)."""
    rng = np.random.Generator(np.random.PCG64(np.random.SeedSequence([int(seed), 0x3AE5])))
    fmax = max_frac * REF_MASS * abs(GRAVITY)
    mag = rng.uniform(0.0, fmax, B)
    ang = rng.uniform(0.0, 2.0 * np.pi, B)
    f = np.stack([mag * np.cos(ang), mag * np.sin(ang), rng.uniform(-fmax, fmax, B)], 1)
    tau = rng.uniform(-max_torque, max_torque, (B, 3))
    j0 = rng.integers(0, N, B)
    L = rng.integers(1, max(1, N // 2) + 1, B)
    k = np.arange(N)
    on = np.where((np.arange(B) % 2 == 0)[:, None], True, (k[None] >= j0[:, None]) & (k[None] < (j0 + L)[:, None]))
    force = np.where(on[:, :, None], f[:, None, :], 0.0)
    torque = np.where((np.arange(B) % 2 == 0)[:, None, None], np.broadcast_to(tau[:, None, :], (B, N, 3)), 0.0)
    return force, torque
