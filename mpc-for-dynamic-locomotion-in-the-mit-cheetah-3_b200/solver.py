"""Python front-ends over the C ABI.

* :class:`BatchedMPC` - tensor API: B independent MPC QPs per call, device tensors in,
  device tensors out (``cmpc_solve``), or host arrays in/out (``cmpc_solve_host``).
* :class:`MPC` - drop-in for the reference's ``MPC`` class (reference ``src/mpc.py:8-318``):
  same constructor, same ``solve(t, logger)`` return dict and attributes, same logger
  calls, same ``RuntimeError`` when the solver does not report "solved".

PyTorch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _capi
from .assembly import assemble_tick, desired_trajectory, pack_problem, reference_velocity
from .gait import GaitPlan, LEGS

STATUS_SOLVED = 1


@dataclass
class SolveStats:
    iters: object
    pri_res: object
    dua_res: object
    status: object


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _np_ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


class BatchedMPC:
    """B independent convex-MPC QPs per call on one GPU.

    Keyword overrides map one-to-one onto ``struct cmpc_config`` (include/cmpc.h):
    ``rho, sigma, alpha, eps_abs, eps_rel, max_iter, check_every, refresh_every, warm_mode,
    r_weight, f_min, f_max, dt, mass, w, ibody_inv``.
    """

    def __init__(self, N=10, max_batch=4096, device=0, **overrides):
        self.N = int(N)
        self.max_batch = int(max_batch)
        cfg = _capi.default_config(self.N, self.max_batch)
        cfg.device = int(device)
        for k, v in overrides.items():
            if k in ("w", "ibody_inv"):
                arr = getattr(cfg, k)
                for i, x in enumerate(v):
                    arr[i] = float(x)
            elif hasattr(cfg, k):
                setattr(cfg, k, type(getattr(cfg, k))(v))
            else:
                raise TypeError(f"unknown solver option {k!r}")
        self.cfg = cfg
        self._h = C.c_void_p()
        _capi.check(_capi.lib().cmpc_create(C.byref(cfg), C.byref(self._h)))
        self.device = int(device)

    # -- lifetime ---------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            _capi.lib().cmpc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- device path ------------------------------------------------------------------
    def solve(self, x0, r, mask, x_des, mu, want_X=True, slot0=0, out=None, stream=None):
        """Device tensors in, device tensors out (asynchronous on the current stream).

        x0 [B,13] f32, r [B,N,4,3] f32, mask [B,N] uint8, x_des [B,N+1,13] f32, mu [B] f32.
        Returns (U [B,N,12], X [B,N+1,13] or None, SolveStats of device tensors)."""
        import torch
        B, N = x0.shape[0], self.N
        self._check_inputs(x0, r, mask, x_des, mu, B, torch)
        dev = x0.device
        if out is None:
            out = self.alloc_outputs(B, want_X, dev)
        U, X, iters, pri, dua, status = out
        s = torch.cuda.current_stream(dev).cuda_stream if stream is None else stream
        _capi.check(_capi.lib().cmpc_solve(
            self._h, B, slot0, _ptr(x0), _ptr(r), _ptr(mask), _ptr(x_des), _ptr(mu), _ptr(U),
            _ptr(X), _ptr(iters), _ptr(pri), _ptr(dua), _ptr(status), C.c_void_p(s)))
        return U, X, SolveStats(iters, pri, dua, status)

    def alloc_outputs(self, B, want_X=True, device=None):
        import torch
        dev = torch.device("cuda", self.device) if device is None else device
        N = self.N
        return (torch.empty((B, N, 12), dtype=torch.float32, device=dev),
                torch.empty((B, N + 1, 13), dtype=torch.float32, device=dev) if want_X else None,
                torch.empty((B,), dtype=torch.int32, device=dev),
                torch.empty((B,), dtype=torch.float32, device=dev),
                torch.empty((B,), dtype=torch.float32, device=dev),
                torch.empty((B,), dtype=torch.int32, device=dev))

    def _check_inputs(self, x0, r, mask, x_des, mu, B, torch):
        N = self.N
        exp = ((x0, (B, 13), torch.float32), (r, (B, N, 4, 3), torch.float32),
               (mask, (B, N), torch.uint8), (x_des, (B, N + 1, 13), torch.float32),
               (mu, (B,), torch.float32))
        for t, shp, dt in exp:
            if tuple(t.shape) != shp or t.dtype != dt or not t.is_contiguous() or not t.is_cuda:
                raise ValueError(f"expected contiguous CUDA {dt} tensor of shape {shp}, got "
                                 f"{tuple(t.shape)} {t.dtype} cuda={t.is_cuda}")
            if t.device.index != self.device:
                raise ValueError(f"tensor on cuda:{t.device.index}, but this solver lives on cuda:{self.device}")

    def condense(self, x0, r, mask, x_des):
        """Dense condensed QP (H [B,12N,12N], g [B,12N]) as device tensors."""
        import torch
        B, N = x0.shape[0], self.N
        H = torch.empty((B, 12 * N, 12 * N), dtype=torch.float32, device=x0.device)
        g = torch.empty((B, 12 * N), dtype=torch.float32, device=x0.device)
        s = torch.cuda.current_stream(x0.device).cuda_stream
        _capi.check(_capi.lib().cmpc_condense(self._h, B, _ptr(x0), _ptr(r), _ptr(mask),
                                              _ptr(x_des), _ptr(H), _ptr(g), C.c_void_p(s)))
        return H, g

    # -- host path --------------------------------------------------------------------
    def solve_host(self, x0, r, mask, x_des, mu, want_X=True, slot0=0, out=None):
        """numpy arrays in (fp32 / uint8, C-contiguous), numpy arrays out; synchronous.
        The C library stages through pinned memory and overlaps copies with the solve."""
        B, N = x0.shape[0], self.N
        for a, dt in ((x0, np.float32), (r, np.float32), (mask, np.uint8), (x_des, np.float32),
                      (mu, np.float32)):
            if a.dtype != dt or not a.flags.c_contiguous:
                raise ValueError("solve_host needs C-contiguous fp32 / uint8 arrays")
        if out is None:
            out = (np.empty((B, N, 12), np.float32),
                   np.empty((B, N + 1, 13), np.float32) if want_X else None,
                   np.empty((B,), np.int32), np.empty((B,), np.float32),
                   np.empty((B,), np.float32), np.empty((B,), np.int32))
        U, X, iters, pri, dua, status = out
        _capi.check(_capi.lib().cmpc_solve_host(
            self._h, B, slot0, _np_ptr(x0), _np_ptr(r), _np_ptr(mask), _np_ptr(x_des), _np_ptr(mu),
            _np_ptr(U), _np_ptr(X), _np_ptr(iters), _np_ptr(pri), _np_ptr(dua), _np_ptr(status)))
        return U, X, SolveStats(iters, pri, dua, status)

    def solve_host_async(self, x0, r, mask, x_des, mu, out, slot0=0):
        """``cmpc_solve_host_async``: page-locked numpy arrays in and out (``out`` = (U, X or None, iters,
        pri_res, dua_res, status), all page-locked); returns a ticket.  The arrays belong to the library until
        ``host_wait(ticket)`` returns; submissions are processed in order (double-buffer to overlap the host
        work of one batch with the device work of the previous one)."""
        B = x0.shape[0]
        for a, dt in ((x0, np.float32), (r, np.float32), (mask, np.uint8), (x_des, np.float32),
                      (mu, np.float32)):
            if a.dtype != dt or not a.flags.c_contiguous:
                raise ValueError("solve_host_async needs C-contiguous fp32 / uint8 arrays")
        U, X, iters, pri, dua, status = out
        ticket = C.c_int32(-1)
        _capi.check(_capi.lib().cmpc_solve_host_async(
            self._h, B, slot0, _np_ptr(x0), _np_ptr(r), _np_ptr(mask), _np_ptr(x_des), _np_ptr(mu),
            _np_ptr(U), _np_ptr(X), _np_ptr(iters), _np_ptr(pri), _np_ptr(dua), _np_ptr(status),
            C.byref(ticket)))
        return int(ticket.value)

    def host_wait(self, ticket):
        _capi.check(_capi.lib().cmpc_host_wait(self._h, int(ticket)))

    # -- warm-start state ---------------------------------------------------------------
    def reset_warm_async(self, B=None, slot0=0, slot_mask=None, stream=None):
        """Stream-ordered reset of slots [slot0, slot0+B); `slot_mask` = uint8 device tensor of B bytes."""
        import torch
        B = self.max_batch - slot0 if B is None else B
        s = torch.cuda.current_stream(torch.device("cuda", self.device)).cuda_stream if stream is None else stream
        _capi.check(_capi.lib().cmpc_reset_warm_async(self._h, B, slot0, _ptr(slot_mask), C.c_void_p(s)))

    def reset_warm(self, slot_mask=None):
        if slot_mask is None:
            _capi.check(_capi.lib().cmpc_reset_warm(self._h, None))
        else:
            m = np.ascontiguousarray(slot_mask, dtype=np.uint8)
            if m.shape != (self.max_batch,):
                raise ValueError("slot_mask must have max_batch entries")
            _capi.check(_capi.lib().cmpc_reset_warm(self._h, _np_ptr(m)))

    def get_warm(self, B, slot0=0):
        import torch
        dev = torch.device("cuda", self.device)
        x = torch.empty((B, self.N, 12), dtype=torch.float32, device=dev)
        y = torch.empty((B, self.N, 4, 3), dtype=torch.float32, device=dev)
        s = torch.cuda.current_stream(dev).cuda_stream
        _capi.check(_capi.lib().cmpc_get_warm(self._h, B, slot0, _ptr(x), _ptr(y), C.c_void_p(s)))
        return x, y

    def set_warm(self, x, y=None, slot0=0):
        import torch
        s = torch.cuda.current_stream(x.device).cuda_stream
        _capi.check(_capi.lib().cmpc_set_warm(self._h, x.shape[0], slot0, _ptr(x), _ptr(y),
                                              C.c_void_p(s)))

    def set_body(self, mass, ibody_inv, slot0=0, stream=None):
        """Rigid bodies of slots [slot0, slot0+B) (``cmpc_set_body``): mass [B] fp32 (kg) and the body-frame
        inverse inertia ibody_inv [B,3,3] fp32, or [B,3] for diagonal ones, CUDA tensors on this solver's device.
        Stream-ordered, no host synchronisation (usable inside a graph capture).  Every later solve of a slot,
        and condense / plant step of problem i = slot i, uses that slot's body; slots never set keep the
        configuration's."""
        import torch
        B = mass.shape[0] if mass.dim() == 1 else -1
        if ibody_inv.dim() == 2 and tuple(ibody_inv.shape) == (B, 3):
            ibody_inv = torch.diag_embed(ibody_inv)
        for t, shp in ((mass, (B,)), (ibody_inv, (B, 3, 3))):
            if tuple(t.shape) != shp or t.dtype != torch.float32 or not t.is_contiguous() or not t.is_cuda:
                raise ValueError(f"expected contiguous CUDA {torch.float32} tensor of shape {shp}, got "
                                 f"{tuple(t.shape)} {t.dtype} cuda={t.is_cuda}")
            if t.device.index != self.device:
                raise ValueError(f"tensor on cuda:{t.device.index}, but this solver lives on cuda:{self.device}")
        s = torch.cuda.current_stream(mass.device).cuda_stream if stream is None else stream
        self._body = (mass, ibody_inv)     # diag_embed's result must live until the copy has run
        _capi.check(_capi.lib().cmpc_set_body(self._h, B, slot0, _ptr(mass), _ptr(ibody_inv), C.c_void_p(s)))

    def set_contact(self, normal, mu, f_min=None, f_max=None, slot0=0, stream=None):
        """Contact surfaces of slots [slot0, slot0+B) (``cmpc_set_contact``): the outward ground normal under each
        leg at each stage, broadcastable to [B,N,4,3] (e.g. one incline per problem, [B,1,1,3]), and the friction
        coefficient mu and normal-force bounds f_min, f_max, broadcastable to [B,N,4] (None = the configuration's
        bounds); fp32 CUDA tensors on this solver's device.  Each force is kept in the friction frustum of its
        surface.  Stream-ordered; the first call of a handle allocates and synchronises, so it must not be
        captured in a CUDA graph, later calls may be.  Slots never set keep flat ground, the solve's mu and the
        configuration's bounds."""
        import torch
        N = self.N
        dev = normal.device
        if f_min is None:
            f_min = torch.full((1, 1, 1), float(self.cfg.f_min), dtype=torch.float32, device=dev)
        if f_max is None:
            f_max = torch.full((1, 1, 1), float(self.cfg.f_max), dtype=torch.float32, device=dev)
        for t in (normal, mu, f_min, f_max):
            if t.dtype != torch.float32 or not t.is_cuda:
                raise ValueError(f"expected CUDA {torch.float32} tensors, got {t.dtype} cuda={t.is_cuda}")
            if t.device.index != self.device:
                raise ValueError(f"tensor on cuda:{t.device.index}, but this solver lives on cuda:{self.device}")
        if normal.dim() == 0 or normal.shape[-1] != 3:
            raise ValueError(f"normal must end in a dimension of 3, got shape {tuple(normal.shape)}")
        try:
            shape = torch.broadcast_shapes(normal.shape[:-1], mu.shape, f_min.shape, f_max.shape, (1, N, 4))
        except RuntimeError as e:
            raise ValueError(f"shapes do not broadcast to [B,{N},4]: {e}") from None
        if len(shape) != 3 or tuple(shape[1:]) != (N, 4):
            raise ValueError(f"shapes broadcast to {tuple(shape)}, not [B,{N},4]")
        B = shape[0]
        normal = normal.expand(B, N, 4, 3).contiguous()
        mu, f_min, f_max = (t.expand(B, N, 4).contiguous() for t in (mu, f_min, f_max))
        s = torch.cuda.current_stream(dev).cuda_stream if stream is None else stream
        self._contact = (normal, mu, f_min, f_max)     # the broadcast copies must live until the copy has run
        _capi.check(_capi.lib().cmpc_set_contact(self._h, B, slot0, _ptr(normal), _ptr(mu), _ptr(f_min),
                                                 _ptr(f_max), C.c_void_p(s)))

    def set_weights(self, w, r_weight=None, slot0=0, stream=None):
        """Cost weights of slots [slot0, slot0+B) (``cmpc_set_weights``): the state weights w [B,13] in the layout
        of the configuration's ``w``, and the force weight r_weight broadcastable to [B] (None = the
        configuration's); fp32 CUDA tensors on this solver's device.  Every later solve of a slot, and condense of
        problem i = slot i, uses that slot's weights.  Stream-ordered; the first call of a handle allocates and
        synchronises, so it must not be captured in a CUDA graph, later calls may be.  Slots never set keep the
        configuration's weights."""
        import torch
        dev = w.device
        if r_weight is None:
            r_weight = torch.full((1,), float(self.cfg.r_weight), dtype=torch.float32, device=dev)
        for t in (w, r_weight):
            if t.dtype != torch.float32 or not t.is_cuda:
                raise ValueError(f"expected CUDA {torch.float32} tensors, got {t.dtype} cuda={t.is_cuda}")
            if t.device.index != self.device:
                raise ValueError(f"tensor on cuda:{t.device.index}, but this solver lives on cuda:{self.device}")
        if w.dim() != 2 or w.shape[1] != 13:
            raise ValueError(f"w must have shape [B,13], got {tuple(w.shape)}")
        B = w.shape[0]
        try:
            r_weight = r_weight.expand(B).contiguous()
        except RuntimeError:
            raise ValueError(f"r_weight of shape {tuple(r_weight.shape)} does not broadcast to [{B}]") from None
        w = w.contiguous()
        s = torch.cuda.current_stream(dev).cuda_stream if stream is None else stream
        self._weights = (w, r_weight)     # the broadcast copies must live until the store has run
        _capi.check(_capi.lib().cmpc_set_weights(self._h, B, slot0, _ptr(w), _ptr(r_weight), C.c_void_p(s)))

    def set_stage_weights(self, w, r_weight=None, slot0=0, stream=None):
        """Stage weights of slots [slot0, slot0+B) (``cmpc_set_stage_weights``): the state weights of every stage,
        broadcastable to [B,N,13] in the layout of the configuration's ``w`` (e.g. one row per robot, [B,1,13], or
        one profile for all robots, [1,N,13]); row i weighs the predicted state X[:, i+1], row N-1 is the terminal
        weight.  r_weight broadcastable to [B] (None = the configuration's); fp32 CUDA tensors on this solver's
        device.  Every later solve of a slot, and condense of problem i = slot i, uses that slot's stage weights, and
        a later ``set_weights`` writes its row into every stage.  Stream-ordered; the first call of a handle
        allocates and synchronises, so it must not be captured in a CUDA graph, later calls may be.  The same row on
        every stage gives the answers of ``set_weights`` with that row bit for bit."""
        import torch
        N = self.N
        dev = w.device
        if r_weight is None:
            r_weight = torch.full((1,), float(self.cfg.r_weight), dtype=torch.float32, device=dev)
        for t in (w, r_weight):
            if t.dtype != torch.float32 or not t.is_cuda:
                raise ValueError(f"expected CUDA {torch.float32} tensors, got {t.dtype} cuda={t.is_cuda}")
            if t.device.index != self.device:
                raise ValueError(f"tensor on cuda:{t.device.index}, but this solver lives on cuda:{self.device}")
        if w.dim() != 3 or w.shape[2] != 13 or w.shape[1] not in (1, N):
            raise ValueError(f"w must broadcast to [B,{N},13] from [B,1,13], [B,{N},13] or [1,{N},13], "
                             f"got {tuple(w.shape)}")
        try:
            B = torch.broadcast_shapes(w.shape[:1], r_weight.shape)[-1]
            w = w.expand(B, N, 13).contiguous()
            r_weight = r_weight.expand(B).contiguous()
        except RuntimeError:
            raise ValueError(f"w {tuple(w.shape)} and r_weight {tuple(r_weight.shape)} do not broadcast to "
                             f"[B,{N},13] and [B]") from None
        s = torch.cuda.current_stream(dev).cuda_stream if stream is None else stream
        self._stage_weights = (w, r_weight)     # the broadcast copies must live until the store has run
        _capi.check(_capi.lib().cmpc_set_stage_weights(self._h, B, slot0, _ptr(w), _ptr(r_weight), C.c_void_p(s)))

    def set_wrench(self, force, torque=None, slot0=0, stream=None):
        """Known external wrenches of slots [slot0, slot0+B) (``cmpc_set_wrench``): the world-frame force on the trunk
        and torque about the CoM at each stage, broadcastable to [B,N,3] (e.g. a constant wrench per robot, [B,1,3];
        torque None = zero); fp32 CUDA tensors on this solver's device.  Every later solve of a slot, and condense /
        plant step of problem i = slot i (the plant applies stage 0), uses that slot's wrench.  Stream-ordered; the
        first call of a handle allocates and synchronises, so it must not be captured in a CUDA graph, later calls
        may be.  Slots never set have zero wrench."""
        import torch
        N = self.N
        dev = force.device
        if torque is None:
            torque = torch.zeros((1, 1, 3), dtype=torch.float32, device=dev)
        for t in (force, torque):
            if t.dtype != torch.float32 or not t.is_cuda:
                raise ValueError(f"expected CUDA {torch.float32} tensors, got {t.dtype} cuda={t.is_cuda}")
            if t.device.index != self.device:
                raise ValueError(f"tensor on cuda:{t.device.index}, but this solver lives on cuda:{self.device}")
        try:
            shape = torch.broadcast_shapes(force.shape, torque.shape, (1, N, 3))
        except RuntimeError as e:
            raise ValueError(f"shapes do not broadcast to [B,{N},3]: {e}") from None
        if len(shape) != 3 or tuple(shape[1:]) != (N, 3):
            raise ValueError(f"shapes broadcast to {tuple(shape)}, not [B,{N},3]")
        B = shape[0]
        force, torque = (t.expand(B, N, 3).contiguous() for t in (force, torque))
        s = torch.cuda.current_stream(dev).cuda_stream if stream is None else stream
        self._wrench = (force, torque)     # the broadcast copies must live until the store has run
        _capi.check(_capi.lib().cmpc_set_wrench(self._h, B, slot0, _ptr(force), _ptr(torque), C.c_void_p(s)))

    def set_force_ref(self, f_ref, weight, slot0=0, stream=None):
        """Force references of slots [slot0, slot0+B) (``cmpc_set_force_ref``): the ground-reaction force wanted from
        each leg at each stage, world frame, broadcastable to [B,N,4,3] (e.g. one per robot and leg, [B,1,4,3]), and
        its weight w_f >= 0, broadcastable to [B,N,4]; fp32 CUDA tensors on this solver's device.  Each stance force
        adds w_f ||f - f_ref||^2 to the objective.  Every later solve of a slot, and condense of problem i = slot i,
        uses that slot's references.  Stream-ordered; the first call of a handle allocates and synchronises, so it
        must not be captured in a CUDA graph, later calls may be.  Slots never set have zero weight, which gives the
        answers of no reference bit for bit."""
        import torch
        N = self.N
        dev = f_ref.device
        for t in (f_ref, weight):
            if t.dtype != torch.float32 or not t.is_cuda:
                raise ValueError(f"expected CUDA {torch.float32} tensors, got {t.dtype} cuda={t.is_cuda}")
            if t.device.index != self.device:
                raise ValueError(f"tensor on cuda:{t.device.index}, but this solver lives on cuda:{self.device}")
        if f_ref.dim() == 0 or f_ref.shape[-1] != 3:
            raise ValueError(f"f_ref must end in a dimension of 3, got shape {tuple(f_ref.shape)}")
        try:
            shape = torch.broadcast_shapes(f_ref.shape[:-1], weight.shape, (1, N, 4))
        except RuntimeError as e:
            raise ValueError(f"shapes do not broadcast to [B,{N},4]: {e}") from None
        if len(shape) != 3 or tuple(shape[1:]) != (N, 4):
            raise ValueError(f"shapes broadcast to {tuple(shape)}, not [B,{N},4]")
        B = shape[0]
        f_ref = f_ref.expand(B, N, 4, 3).contiguous()
        weight = weight.expand(B, N, 4).contiguous()
        s = torch.cuda.current_stream(dev).cuda_stream if stream is None else stream
        self._force_ref = (f_ref, weight)     # the broadcast copies must live until the store has run
        _capi.check(_capi.lib().cmpc_set_force_ref(self._h, B, slot0, _ptr(f_ref), _ptr(weight), C.c_void_p(s)))

    def cache_meta(self, B, slot0=0):
        """[B,4] device tensor {rho, yaw, valid, reused-by-last-solve} of the factorisation cache."""
        import torch
        out = torch.empty((B, 4), dtype=torch.float32, device=torch.device("cuda", self.device))
        s = torch.cuda.current_stream(out.device).cuda_stream
        _capi.check(_capi.lib().cmpc_get_cache_meta(self._h, B, slot0, _ptr(out), C.c_void_p(s)))
        return out

    @property
    def last_kernel_ms(self) -> float:
        """Duration of the solve kernel of the last :meth:`solve` (needs ``time_kernel=1``)."""
        v = C.c_float()
        _capi.check(_capi.lib().cmpc_last_kernel_ms(self._h, C.byref(v)))
        return float(v.value)

    @property
    def launch_count(self) -> int:
        return int(_capi.lib().cmpc_launch_count(self._h))


class MPC:
    """Drop-in replacement of the reference's ``MPC`` (reference ``src/mpc.py:8-318``).

    ``MPC(lite3, initial, footstep_planner, params).solve(t, logger)`` returns
    ``{'FL_FOOT': f(3,), 'FR_FOOT': ..., 'HL_FOOT': ..., 'HR_FOOT': ...}`` (float64, world
    frame, forces on the robot) and keeps the reference's attributes ``x, x_log, x_plot, u,
    u_plot, com_pos_start, yaw_start``.  The QP of every tick is solved on the GPU through
    ``cmpc_solve_host`` with the reference's warm-start semantics (previous primal solution,
    unshifted; zero duals)."""

    def __init__(self, lite3, initial, footstep_planner, params, **solver_options):
        self.params = params
        self.lite3 = lite3
        self.N = params["N"]
        self.delta = params["world_time_step"]
        self.h = params["h"]
        self.mu = params["µ"] if "µ" in params else params["μ"]   # U+00B5 (reference) or U+03BC
        self.initial = initial
        self.footstep_planner = footstep_planner
        self.com_pos_start = initial["com_position"]     # aliased and mutated, src/mpc.py:36-37
        self.com_pos_start[2] = self.h
        self.yaw_start = initial["yaw"]
        self.m = 8.885                                    # src/mpc.py:71
        opts = dict(dt=self.delta, warm_mode=1)
        opts.update(solver_options)
        self.solver = BatchedMPC(N=self.N, max_batch=1, **opts)

    def _plan(self):
        fp = self.footstep_planner
        if isinstance(fp, GaitPlan):
            return fp
        return GaitPlan.from_reference_planner(fp, self.params.get("step_height", 0.08))

    def solve(self, t, logger):
        plan = self._plan()
        v_com_gait, omega = reference_velocity(plan, t, self.params)         # src/mpc.py:178-183
        current_state = self.lite3.retrieve_state()                           # src/mpc.py:190-198
        state_rpy = np.array([current_state["TORSO"]["pos"]]).T
        state_com = np.array([current_state["com"]["pos"]]).T
        state_av = np.array([current_state["TORSO"]["vel"]]).T
        state_lv = np.array([current_state["com"]["vel"]]).T
        self.x = np.vstack([state_rpy, state_com, state_av, state_lv, self.params["g"]])
        x_des_num = desired_trajectory(self.N, self.delta, self.initial["roll"],
                                       self.initial["pitch"], self.yaw_start, self.com_pos_start,
                                       v_com_gait, omega, self.params["g"])
        feet = np.stack([np.asarray(current_state[leg]["pos"][3:], dtype=float) for leg in LEGS])
        r, stance = assemble_tick(plan, t, self.N, self.delta, self.x[:, 0], feet, x_des_num)
        x0f, rf, maskf, xdf = pack_problem(self.x[:, 0], r, stance, x_des_num)
        U, X, stats = self.solver.solve_host(
            x0f[None], rf[None], maskf[None], xdf[None], np.array([self.mu], dtype=np.float32))
        if int(stats.status[0]) != STATUS_SOLVED:                            # CasADi raises too
            raise RuntimeError(f"MPC QP not solved (status {int(stats.status[0])}, "
                               f"{int(stats.iters[0])} iterations)")
        self.com_pos_start += v_com_gait * self.delta                        # src/mpc.py:261-262
        self.yaw_start += omega * self.delta
        Xs = X[0].astype(np.float64).T                                       # (13, N+1)
        Us = U[0].astype(np.float64).T                                       # (12, N)
        self.x_log = Xs[:-1, :]
        self.x_plot = Xs[3:6, :]
        self.u = Us[:, 0].copy()
        self.u_plot = Us
        self.iters = int(stats.iters[0])
        forces = {leg: self.u[3 * i:3 * i + 3] for i, leg in enumerate(LEGS)}
        forces_plot = np.array([self.u_plot[2, :], self.u_plot[5, :], self.u_plot[8, :],
                                self.u_plot[11, :]])
        x_curr = (state_rpy.flatten().tolist() + state_com.flatten().tolist()
                  + state_av.flatten().tolist() + state_lv.flatten().tolist())
        logger.log_tracking_data(x_curr, x_des_num[:-1, 0])                  # src/mpc.py:295
        if t == 0 or t == 80:                                                # src/mpc.py:297-301
            logger.log_mpc_predictions(self.x_log, x_des_num[:-1, :], forces_plot, t)
        return forces

    def update_r_num(self, time, leg_name, next_com):
        """reference ``src/mpc.py:306-318`` (kept for callers that use it directly)."""
        return self._plan().foot_position(time)[LEGS.index(leg_name)] - next_com
