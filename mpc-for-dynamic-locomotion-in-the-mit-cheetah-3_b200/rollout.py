"""Closed-loop, warm-started MPC rollouts of many robots on one GPU (BASELINE config 5).

Every tick runs, entirely on the device:
  ``cmpc_assemble``  -> x_des, lever arms, contact masks of the tick  (reference src/mpc.py:178-255)
  ``cmpc_solve``     -> ground-reaction forces, warm-started from the previous tick with the
                        reference's semantics (previous primal solution unshifted, zero duals,
                        src/mpc.py:270-271)
  ``cmpc_plant_step``-> single-rigid-body forward-Euler plant with the applied first-stage
                        forces (DART, the reference's simulator, is not available; the plant
                        is the model the MPC itself predicts with), reference accumulators,
                        tick counter
The per-tick launch sequence is static (the tick lives in device memory), so it can be
captured once in a CUDA graph and replayed.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi
from .gait import GAITS
from .problems import BatchedGaitPlan, NOMINAL_COM, NOMINAL_FEET, GRAVITY, DT
from .solver import BatchedMPC, _ptr


class ClosedLoopRollout:
    def __init__(self, B, N=10, gaits=("trot",), mu=(0.3, 1.0), seed=0, total_steps=20, device=0,
                 v_scale=1.0, mass=None, ibody_inv=None, w=None, r_weight=None, force=None, torque=None,
                 f_ref=None, f_weight=None, w_stage=None, **solver_options):
        """`mass` (B,) and `ibody_inv` (B,3,3) or (B,3), numpy: per-robot bodies, set once here; the plant
        integrates each robot with the body its controller predicts with.  None: the configuration's.
        `w` (B,13) and `r_weight` (B,) or None, numpy: per-robot cost weights (BatchedMPC.set_weights), set once
        here.  None: the configuration's.
        `force` and `torque` (B,3) or (B,N,3), numpy: per-robot known external wrenches, world frame
        (BatchedMPC.set_wrench), set once here; the controller predicts with them over its horizon and the plant
        applies their stage 0 at every tick.  None: zero.
        `f_ref` (B,4,3) or (B,N,4,3) and `f_weight` (B,), (B,4) or (B,N,4), numpy: per-robot force references,
        world frame, and their weights (BatchedMPC.set_force_ref), set once here, the same at every tick (a (B,4,3)
        reference and a (B,) or (B,4) weight hold for every stage).  None: no reference.
        `w_stage` (B,N,13) or (N,13), numpy: per-robot stage weights (BatchedMPC.set_stage_weights; row i weighs the
        predicted state i + 1, row N-1 is the terminal weight), with `r_weight` as above, set once here; an (N,13)
        profile holds for every robot.  Not together with `w`.  None: no stage weights."""
        import torch
        self.torch = torch
        self.B, self.N = int(B), int(N)
        rng = np.random.default_rng(seed)
        gid = rng.integers(0, len(gaits), size=B)
        table = [GAITS[g] for g in gaits]
        first_swing = np.array([table[i][0] for i in gid], dtype=np.int64)
        ss = np.array([table[i][1] for i in gid], dtype=np.int64)
        ds = np.array([table[i][2] for i in gid], dtype=np.int64)
        v_ref = np.stack([np.array([table[i][3] for i in gid]) * v_scale, np.zeros(B), np.zeros(B)], 1)
        om_ref = np.zeros(B)
        self.plan = BatchedGaitPlan.build(NOMINAL_FEET, np.zeros(B), first_swing, ss, ds, v_ref, om_ref,
                                          total_steps=total_steps)
        self.mu_host = np.linspace(mu[0], mu[1], B)                       # friction sweep
        dev = torch.device("cuda", device)
        self.dev = dev
        f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
        self.plan_pos = f32(self.plan.pos)
        bits = (self.plan.feet_id * np.array([1, 2, 4, 8])).sum(-1).astype(np.uint8)
        self.feet_id = torch.from_numpy(np.ascontiguousarray(bits)).to(dev)
        self.ss = torch.from_numpy(ss.astype(np.int32)).to(dev)
        self.ds = torch.from_numpy(ds.astype(np.int32)).to(dev)
        self.v_ref, self.omega_ref = f32(v_ref), f32(om_ref)
        self.rp0 = torch.zeros((B, 2), dtype=torch.float32, device=dev)
        self.mu = f32(self.mu_host)
        x0 = np.zeros((B, 13))
        x0[:, 3:6] = NOMINAL_COM
        x0[:, 12] = GRAVITY
        self.x = f32(x0)
        self.yaw_start = torch.zeros(B, dtype=torch.float32, device=dev)
        self.com_start = f32(np.tile(NOMINAL_COM, (B, 1)))
        self.tick = torch.zeros(1, dtype=torch.int32, device=dev)
        self.track_err = torch.zeros((B, 2), dtype=torch.float32, device=dev)
        self.x_des = torch.empty((B, N + 1, 13), dtype=torch.float32, device=dev)
        self.r = torch.empty((B, N, 4, 3), dtype=torch.float32, device=dev)
        self.mask = torch.empty((B, N), dtype=torch.uint8, device=dev)
        # closed-loop defaults: reference warm start; no hardest-first scheduling (warm-started ticks
        # have uniform iteration counts: the two scheduling kernels only cost time, measured 0.372 ->
        # 0.355 ms per tick); factorisation cache (standing phases reuse -P^-1: 0.355 -> 0.295 ms)
        opts = dict(warm_mode=1, lpt_schedule=0, cache_factorization=1 if self.N in (10, 30) else 0)
        opts.update(solver_options)
        self.mpc = BatchedMPC(N=N, max_batch=B, device=device, **opts)
        self.out = self.mpc.alloc_outputs(B, want_X=False, device=dev)
        if (mass is None) != (ibody_inv is None):
            raise ValueError("mass and ibody_inv go together")
        if mass is not None:
            ib = np.asarray(ibody_inv, dtype=np.float64)
            if ib.shape == (B, 3):
                ib = ib[:, None, :] * np.eye(3)
            if np.shape(mass) != (B,) or ib.shape != (B, 3, 3):
                raise ValueError("mass must be (B,) and ibody_inv (B,3,3) or (B,3)")
            self.body = (f32(mass), f32(ib))
            self.mpc.set_body(*self.body)
        if r_weight is not None and w is None and w_stage is None:
            raise ValueError("r_weight needs w or w_stage")
        if w is not None and w_stage is not None:
            raise ValueError("w and w_stage are two forms of the state weights: give one")
        if w_stage is not None:
            ws = np.asarray(w_stage, dtype=np.float64)
            if ws.shape == (N, 13):
                ws = np.broadcast_to(ws, (B, N, 13))
            if ws.shape != (B, N, 13) or (r_weight is not None and np.shape(r_weight) != (B,)):
                raise ValueError("w_stage must be (B,N,13) or (N,13) and r_weight (B,)")
            self.stage_weights = (f32(ws), None if r_weight is None else f32(r_weight))
            self.mpc.set_stage_weights(*self.stage_weights)
        if w is not None:
            if np.shape(w) != (B, 13) or (r_weight is not None and np.shape(r_weight) != (B,)):
                raise ValueError("w must be (B,13) and r_weight (B,)")
            self.weights = (f32(w), None if r_weight is None else f32(r_weight))
            self.mpc.set_weights(*self.weights)
        if force is not None or torque is not None:
            def wrench(a):
                a = np.zeros((B, 1, 3)) if a is None else np.asarray(a, dtype=np.float64)
                if a.shape == (B, 3):
                    a = a[:, None, :]
                if a.shape not in ((B, 1, 3), (B, N, 3)):
                    raise ValueError("force and torque must be (B,3) or (B,N,3)")
                return f32(a)
            self.wrench = (wrench(force), wrench(torque))
            self.mpc.set_wrench(*self.wrench)
        if (f_ref is None) != (f_weight is None):
            raise ValueError("f_ref and f_weight go together")
        if f_ref is not None:
            fr = np.asarray(f_ref, dtype=np.float64)
            fw = np.asarray(f_weight, dtype=np.float64)
            if fr.shape == (B, 4, 3):
                fr = fr[:, None]
            if fw.shape == (B,):
                fw = fw[:, None, None]
            elif fw.shape == (B, 4):
                fw = fw[:, None, :]
            if fr.shape not in ((B, 1, 4, 3), (B, N, 4, 3)) or fw.shape not in ((B, 1, 1), (B, 1, 4), (B, N, 4)):
                raise ValueError("f_ref must be (B,4,3) or (B,N,4,3) and f_weight (B,), (B,4) or (B,N,4)")
            self.force_ref = (f32(fr), f32(fw))
            self.mpc.set_force_ref(*self.force_ref)
        self.gt = _capi.GaitTables(
            plan_pos=self.plan_pos.data_ptr(), feet_id=self.feet_id.data_ptr(), ss=self.ss.data_ptr(),
            ds=self.ds.data_ptr(), v_ref=self.v_ref.data_ptr(), omega_ref=self.omega_ref.data_ptr(),
            rp0=self.rp0.data_ptr(), S=self.plan.n_steps, total_steps=total_steps,
            step_height=float(self.plan.step_height), g=GRAVITY)
        self.acc = torch.zeros(3, dtype=torch.int64, device=dev)   # iterations, unsolved, cache hits
        self._graph = None

    # one tick on the current stream -----------------------------------------------------
    def step(self, stream=None):
        torch, L, h = self.torch, _capi.lib(), self.mpc._h
        s = C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream if stream is None else stream)
        _capi.check(L.cmpc_assemble(h, self.B, C.byref(self.gt), _ptr(self.tick), _ptr(self.x),
                                    _ptr(self.yaw_start), _ptr(self.com_start), _ptr(self.x_des),
                                    _ptr(self.r), _ptr(self.mask), s))
        self.mpc.solve(self.x, self.r, self.mask, self.x_des, self.mu, want_X=False, out=self.out,
                       stream=s.value)
        _capi.check(L.cmpc_plant_step(h, self.B, C.byref(self.gt), _ptr(self.tick), _ptr(self.x),
                                      _ptr(self.r), _ptr(self.out[0]), _ptr(self.x_des),
                                      _ptr(self.yaw_start), _ptr(self.com_start),
                                      _ptr(self.track_err), s))

    def accumulate_stats(self):
        s = C.c_void_p(self.torch.cuda.current_stream(self.dev).cuda_stream)
        _capi.check(_capi.lib().cmpc_accumulate_stats(self.mpc._h, self.B, 0, _ptr(self.out[2]),
                                                      _ptr(self.out[5]), _ptr(self.acc), s))

    def capture(self, ticks_per_graph=10):
        """Capture `ticks_per_graph` ticks in a CUDA graph (static launch sequence)."""
        torch = self.torch
        self.step()
        torch.cuda.synchronize(self.dev)                      # warm-up outside capture
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(ticks_per_graph):
                self.step()
                self.accumulate_stats()
        self._graph, self._tpg = g, ticks_per_graph
        return g

    def run(self, ticks, use_graph=True, ticks_per_graph=10):
        """Advance all robots by `ticks` ticks.  Returns the number of ticks executed."""
        done = 0
        if use_graph:
            if self._graph is None:
                self.capture(ticks_per_graph)
                done += 1
            while done + self._tpg <= ticks:
                self._graph.replay()
                done += self._tpg
        while done < ticks:
            self.step()
            self.accumulate_stats()
            done += 1
        return done

    def summary(self):
        self.torch.cuda.synchronize(self.dev)
        t = int(self.tick.item())
        x = self.x.cpu().numpy()
        te = self.track_err.cpu().numpy() / max(t, 1)
        return dict(ticks=t, com_z_min=float(x[:, 5].min()), com_z_max=float(x[:, 5].max()),
                    rms_pos_err=float(np.sqrt(te[:, 0].mean())), rms_ang_err=float(np.sqrt(te[:, 1].mean())),
                    mean_iters=float(self.acc[0].item()) / max(t * self.B, 1),
                    cache_hit_frac=float(self.acc[2].item()) / max(t * self.B, 1),
                    unsolved=int(self.acc[1].item()), finite=bool(np.isfinite(x).all()))
