"""CPU-side checks of the C ABI: the shared library loads, exports every symbol that
include/cmpc.h declares, its config struct matches the ctypes mirror, and - with no GPU -
it fails loudly instead of falling back to a CPU path."""
import ctypes as C
import os
import re

import pytest

import mpc_b200 as pkg
from mpc_b200 import _capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_are_exported():
    hdr = open(os.path.join(ROOT, "include", "cmpc.h")).read()
    declared = set(re.findall(r"\b(cmpc_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"cmpc_config", "cmpc_handle"}
    assert declared == set(_capi.SYMBOLS)
    L = _capi.lib()
    for name in declared:
        assert hasattr(L, name), name


def test_default_config_matches_reference_constants():
    cfg = _capi.default_config(10, 4096)
    assert (cfg.N, cfg.max_batch) == (10, 4096)
    assert cfg.dt == pytest.approx(0.01) and cfg.mass == pytest.approx(8.885)      # src/mpc.py:71
    assert list(cfg.ibody_inv) == pytest.approx([1 / 0.24, 1, 1])                  # src/mpc.py:73-76
    assert list(cfg.w) == pytest.approx([1e4, 2.7e4, 1e4, 2.7e5, 2.7e5, 2.7e5, 1e4, 1e4, 1e4,
                                         1.6e4, 1.6e4, 1.6e4, 0])                  # src/mpc.py:121-134
    assert cfg.r_weight == 0.0 and (cfg.f_min, cfg.f_max) == (3.0, 100.0)          # src/mpc.py:45-46,121
    assert cfg.max_iter == 1000                                                    # src/mpc.py:51
    assert cfg.eps_abs == pytest.approx(1e-3) and cfg.eps_rel == pytest.approx(1e-3)
    assert cfg.warm_mode == 1
    assert cfg.rho == pytest.approx(0.5) and cfg.adaptive_rho_tolerance == pytest.approx(3.0)
    c30 = _capi.default_config(30, 8)            # stage-wise kernel: cheap refactorisation, tighter rho tolerance
    assert c30.rho == pytest.approx(1.5) and c30.adaptive_rho_tolerance == pytest.approx(1.5)
    assert _capi.default_config(20, 8).adaptive_rho_tolerance == pytest.approx(1.5)
    assert _capi.default_config(16, 8).adaptive_rho_tolerance == pytest.approx(3.0)
    assert cfg.rho_max == pytest.approx(300.0) and cfg.rho_min == pytest.approx(0.05)
    # struct layout: the C side zero-fills then writes; a mismatch would scramble the tail
    assert cfg.device == 0 and cfg.kernel_variant == 0


def test_supported_horizons_and_version():
    hs = _capi.supported_horizons()
    assert 10 in hs and 30 in hs and hs == sorted(hs)
    assert _capi.lib().cmpc_version() == 3


def test_any_horizon_maps_to_a_compiled_kernel():
    """reference src/main.py:41 accepts any params['N']: horizons without their own kernel run
    padded on the next compiled one."""
    hs = _capi.supported_horizons()
    assert _capi.lib().cmpc_max_horizon() == max(hs) == 60
    for N in range(1, 61):
        k = _capi.kernel_horizon(N)
        assert k in hs and k >= N and not any(N <= h < k for h in hs)
    with pytest.raises(pkg.CmpcError):
        _capi.kernel_horizon(61)
    assert _capi.has_variant(10, 0) and _capi.has_variant(30, 5) and not _capi.has_variant(10, 7)
    assert not _capi.has_variant(10, 1) and not _capi.has_variant(60, 5)


def test_alias_package_is_one_module():
    """`mpc_b200.<sub>` must be the same module objects as the hyphen-named package's."""
    import importlib
    import mpc_b200.gait
    import mpc_b200.solver
    from mpc_b200.gait import GaitPlan
    real = importlib.import_module("mpc-for-dynamic-locomotion-in-the-mit-cheetah-3_b200")
    assert GaitPlan is pkg.GaitPlan is real.gait.GaitPlan
    assert mpc_b200.solver.MPC is pkg.MPC and mpc_b200.solver is real.solver
    assert pkg._capi is real._capi and pkg.CmpcError is real._capi.CmpcError


def test_argument_validation_without_touching_the_gpu():
    L = _capi.lib()
    h = C.c_void_p()
    cfg = _capi.default_config(61, 16)           # beyond the largest compiled kernel
    assert L.cmpc_create(C.byref(cfg), C.byref(h)) == -3
    assert b"N=61" in L.cmpc_last_error()
    cfg = _capi.default_config(10, 16)
    cfg.cache_factorization, cfg.check_every, cfg.refresh_every = 1, 5, 3
    assert L.cmpc_create(C.byref(cfg), C.byref(h)) == -1
    cfg = _capi.default_config(10, 0)
    assert L.cmpc_create(C.byref(cfg), C.byref(h)) == -1
    cfg = _capi.default_config(10, 16)
    cfg.w[7] = 5.0                                # w[6] != w[7]
    assert L.cmpc_create(C.byref(cfg), C.byref(h)) == -3
    cfg = _capi.default_config(10, 16)
    cfg.alpha = 2.5
    assert L.cmpc_create(C.byref(cfg), C.byref(h)) == -1
    assert L.cmpc_destroy(None) == 0


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(pkg.CmpcError) as e:
        pkg.BatchedMPC(N=10, max_batch=8)
    assert e.value.code == -4 and "no CPU fallback" in str(e.value)
