"""ctypes binding of ``csrc/libcmpc.so`` (C ABI declared in ``include/cmpc.h``).

There is no CPU fallback: if the shared library is missing, :func:`lib` raises, and if
no CUDA device is visible ``cmpc_create`` returns ``CMPC_ERR_NO_DEVICE`` which surfaces
as :class:`CmpcError`.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libcmpc.so")
SOURCES = [os.path.join(CSRC, "cmpc.cu"), os.path.join(CSRC, "cmpc_body.cu"), os.path.join(CSRC, "cmpc_contact.cu"),
           os.path.join(CSRC, "cmpc_weights.cu"), os.path.join(CSRC, "cmpc_wrench.cu"),
           os.path.join(CSRC, "cmpc_force.cu"), os.path.join(CSRC, "cmpc_stage.cu")]
HEADERS = [os.path.join(CSRC, "cmpc_kernels.cuh"), os.path.join(CSRC, "cmpc_riccati.cuh"),
           os.path.join(CSRC, "cmpc_tc.cuh"), os.path.join(CSRC, "cmpc_launch.cuh"),
           os.path.join(_ROOT, "include", "cmpc.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]

#: every symbol include/cmpc.h declares
SYMBOLS = ("cmpc_default_config", "cmpc_create", "cmpc_destroy", "cmpc_solve", "cmpc_solve_host",
           "cmpc_solve_host_async", "cmpc_host_wait",
           "cmpc_condense", "cmpc_reset_warm", "cmpc_get_warm", "cmpc_set_warm",
           "cmpc_launch_count", "cmpc_supported_horizons", "cmpc_version", "cmpc_last_error",
           "cmpc_assemble", "cmpc_plant_step", "cmpc_fp32_peak", "cmpc_leg_torques", "cmpc_last_kernel_ms", "cmpc_get_cache_meta", "cmpc_accumulate_stats",
           "cmpc_reset_warm_async", "cmpc_max_horizon", "cmpc_kernel_horizon", "cmpc_has_variant",
           "cmpc_leg_kinematics", "cmpc_set_body", "cmpc_set_contact", "cmpc_set_weights",
           "cmpc_set_wrench", "cmpc_set_force_ref", "cmpc_set_stage_weights")


class CmpcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"cmpc error {code}: {msg}")
        self.code = code


class Config(C.Structure):
    """Mirror of ``struct cmpc_config``."""
    _fields_ = [("N", C.c_int32), ("max_batch", C.c_int32), ("dt", C.c_float), ("mass", C.c_float),
                ("ibody_inv", C.c_float * 3), ("w", C.c_float * 13), ("r_weight", C.c_float),
                ("f_min", C.c_float), ("f_max", C.c_float), ("rho", C.c_float),
                ("sigma", C.c_float), ("alpha", C.c_float), ("eps_abs", C.c_float),
                ("eps_rel", C.c_float), ("max_iter", C.c_int32), ("check_every", C.c_int32),
                ("refresh_every", C.c_int32), ("warm_mode", C.c_int32),
                ("adaptive_rho_interval", C.c_int32), ("adaptive_rho_tolerance", C.c_float),
                ("rho_min", C.c_float), ("rho_max", C.c_float),
                ("kernel_variant", C.c_int32), ("lpt_schedule", C.c_int32),
                ("device", C.c_int32), ("host_zero_copy", C.c_int32), ("cache_factorization", C.c_int32),
                ("cache_tol_r", C.c_float), ("cache_tol_yaw", C.c_float), ("cache_max_iter", C.c_int32),
                ("time_kernel", C.c_int32)]


class GaitTables(C.Structure):
    """Mirror of ``struct cmpc_gait_tables`` (device pointers)."""
    _fields_ = [("plan_pos", C.c_void_p), ("feet_id", C.c_void_p), ("ss", C.c_void_p),
                ("ds", C.c_void_p), ("v_ref", C.c_void_p), ("omega_ref", C.c_void_p),
                ("rp0", C.c_void_p), ("S", C.c_int32), ("total_steps", C.c_int32),
                ("step_height", C.c_float), ("g", C.c_float)]


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(f) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile libcmpc.so in-tree for sm_100a with nvcc (cross-compiles without a GPU)."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH] + SOURCES
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


_lib = None


def lib() -> C.CDLL:
    """Load the library (never builds implicitly on a GPU box: the .so travels in-tree)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CmpcError(-4, f"{LIB_PATH} is missing - run `python -c 'import __graft_entry__ as g; "
                            f"g.build()'`; there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, i32, f32p, u8p, i32p = C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p
    L.cmpc_default_config.argtypes = [C.POINTER(Config), i32, i32]
    L.cmpc_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.cmpc_destroy.argtypes = [vp]
    L.cmpc_solve.argtypes = [vp, i32, i32, f32p, f32p, u8p, f32p, f32p, f32p, f32p, i32p, f32p,
                             f32p, i32p, vp]
    L.cmpc_solve_host.argtypes = [vp, i32, i32, f32p, f32p, u8p, f32p, f32p, f32p, f32p, i32p,
                                  f32p, f32p, i32p]
    L.cmpc_solve_host_async.argtypes = [vp, i32, i32, f32p, f32p, u8p, f32p, f32p, f32p, f32p, i32p,
                                        f32p, f32p, i32p, i32p]
    L.cmpc_host_wait.argtypes = [vp, i32]
    L.cmpc_condense.argtypes = [vp, i32, f32p, f32p, u8p, f32p, f32p, f32p, vp]
    L.cmpc_reset_warm.argtypes = [vp, u8p]
    L.cmpc_reset_warm_async.argtypes = [vp, i32, i32, u8p, vp]
    L.cmpc_max_horizon.argtypes = []
    L.cmpc_kernel_horizon.argtypes = [i32]
    L.cmpc_has_variant.argtypes = [i32, i32]
    L.cmpc_get_warm.argtypes = [vp, i32, i32, f32p, f32p, vp]
    L.cmpc_set_warm.argtypes = [vp, i32, i32, f32p, f32p, vp]
    L.cmpc_set_body.argtypes = [vp, i32, i32, f32p, f32p, vp]
    L.cmpc_set_contact.argtypes = [vp, i32, i32, f32p, f32p, f32p, f32p, vp]
    L.cmpc_set_weights.argtypes = [vp, i32, i32, f32p, f32p, vp]
    L.cmpc_set_wrench.argtypes = [vp, i32, i32, f32p, f32p, vp]
    L.cmpc_set_force_ref.argtypes = [vp, i32, i32, f32p, f32p, vp]
    L.cmpc_set_stage_weights.argtypes = [vp, i32, i32, f32p, f32p, vp]
    gtp = C.POINTER(GaitTables)
    L.cmpc_assemble.argtypes = [vp, i32, gtp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.cmpc_plant_step.argtypes = [vp, i32, gtp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.cmpc_leg_torques.argtypes = [vp, i32, gtp] + [vp] * 9 + [C.POINTER(C.c_float)] * 2 + [vp] * 4
    L.cmpc_leg_kinematics.argtypes = [vp, i32] + [vp] * 12 + [C.c_float, vp]
    L.cmpc_fp32_peak.argtypes = [i32, C.POINTER(C.c_float)]
    L.cmpc_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float)]
    L.cmpc_get_cache_meta.argtypes = [vp, i32, i32, vp, vp]
    L.cmpc_accumulate_stats.argtypes = [vp, i32, i32, vp, vp, vp, vp]
    L.cmpc_launch_count.argtypes = [vp]
    L.cmpc_launch_count.restype = C.c_int64
    L.cmpc_supported_horizons.argtypes = [C.POINTER(C.c_int32), i32]
    L.cmpc_version.restype = C.c_int
    L.cmpc_last_error.restype = C.c_char_p
    for name in SYMBOLS:
        if name not in ("cmpc_launch_count", "cmpc_last_error"):
            getattr(L, name).restype = C.c_int
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != 0:
        raise CmpcError(rc, lib().cmpc_last_error().decode())


def default_config(N: int, max_batch: int) -> Config:
    cfg = Config()
    check(lib().cmpc_default_config(C.byref(cfg), N, max_batch))
    return cfg


def fp32_peak(device=0) -> float:
    """Measured FP32 FMA peak of `device` in TFLOP/s."""
    v = C.c_float()
    check(lib().cmpc_fp32_peak(device, C.byref(v)))
    return float(v.value)


def kernel_horizon(N: int) -> int:
    """Compiled horizon that horizon N runs on (raises CmpcError outside 1..cmpc_max_horizon())."""
    rc = lib().cmpc_kernel_horizon(int(N))
    if rc < 0:
        check(rc)
    return rc


def has_variant(N: int, variant: int) -> bool:
    return bool(lib().cmpc_has_variant(int(N), int(variant)))


def supported_horizons():
    buf = (C.c_int32 * 64)()
    n = lib().cmpc_supported_horizons(buf, 64)
    return [int(buf[i]) for i in range(min(n, 64))]
