"""ctypes binding of include/carmpc.h (``carmpc_b200/_lib/libcarmpc_b200.so``).

This is the only door from Python into the CUDA library.  There is no CPU fallback: if the library is
missing it is built with nvcc (``carmpc_b200.build``); if that is impossible, or a call fails, a
``CarmpcError`` is raised with the library's own message.
"""
from __future__ import annotations

import ctypes
import os

from . import build as _build


class CarmpcError(RuntimeError):
    """A C-ABI call returned a negative status."""


class QPOpts(ctypes.Structure):
    """``carmpc_qp_opts`` (include/carmpc.h)."""
    _fields_ = [("rho", ctypes.c_double), ("alpha", ctypes.c_double), ("eps_abs", ctypes.c_double),
                ("eps_rel", ctypes.c_double), ("eps_prim_inf", ctypes.c_double),
                ("max_iter", ctypes.c_int32), ("check_every", ctypes.c_int32),
                ("scaling_iters", ctypes.c_int32), ("polish", ctypes.c_int32)]


class DisturbanceModel(ctypes.Structure):
    """``carmpc_disturbance_model`` (include/carmpc.h)."""
    _fields_ = [("Bd", ctypes.c_double * 4), ("Cd", ctypes.c_double * 3), ("L1", ctypes.c_double * 12),
                ("L2", ctypes.c_double * 3), ("Bd_plant", ctypes.c_double * 4), ("Cd_plant", ctypes.c_double * 3)]


class LoopNoiseParams(ctypes.Structure):
    """``carmpc_loop_noise`` (include/carmpc.h)."""
    _fields_ = [("seed", ctypes.c_uint64), ("first_run", ctypes.c_int64), ("Lw", ctypes.c_double * 16),
                ("Lv", ctypes.c_double * 16)]


_vp, _dp, _i64, _i32 = ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int

#: name -> (restype, argtypes); every function include/carmpc.h declares
SIGNATURES = {
    "carmpc_last_error": (ctypes.c_char_p, []),
    "carmpc_version": (ctypes.c_char_p, []),
    "carmpc_destroy": (None, [_vp]),
    "carmpc_polytope_create": (_i32, [_dp, _i32, ctypes.POINTER(_vp)]),
    "carmpc_membership_bitset": (_i32, [_vp, _dp, _dp, _dp, _dp, _i64, _vp, _vp, _i32, _vp]),
    "carmpc_polytope_tune": (_i32, [_vp, _dp, _dp, _dp, _dp, _i64, _vp]),
    "carmpc_membership_grid": (_i32, [_vp, _dp, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32),
                                      _vp, _vp, _vp]),
    "carmpc_membership_bitset_host": (_i32, [_vp, _dp, _dp, _dp, _dp, _i64, _vp, ctypes.POINTER(_i64), _i32]),
    "carmpc_rollout_create": (_i32, [_dp, _dp, _dp, _i32, _dp, _dp, _i32, _dp, _i32, _i32, ctypes.POINTER(_vp)]),
    "carmpc_rollout_bitset": (_i32, [_vp, _dp, _dp, _dp, _dp, _i64, _vp, _vp, _vp, _vp]),
    "carmpc_rollout_bitset_host": (_i32, [_vp, _dp, _dp, _dp, _dp, _i64, _vp, _vp, ctypes.POINTER(_i64)]),
    "carmpc_rollout_get_rows": (_i32, [_vp, _dp, _i32]),
    "carmpc_rollout_reduce_screen": (_i32, [_vp, ctypes.POINTER(ctypes.c_int32), _i32, ctypes.POINTER(ctypes.c_int32), _dp, _i32]),
    "carmpc_scan_staging": (_i32, [_vp, _i32, _i32, _i32]),
    "carmpc_shard_create": (_i32, [_i32, _i32, _i64, ctypes.POINTER(_vp)]),
    "carmpc_shard_export": (_i32, [_vp, _vp]),
    "carmpc_shard_connect": (_i32, [_vp, _vp]),
    "carmpc_shard_connect_local": (_i32, [_vp, ctypes.POINTER(_vp)]),
    "carmpc_membership_bitset_sharded": (_i32, [_vp, _vp, _dp, _dp, _dp, _dp, _i64, _i64, _i64, _i32, _vp, _i32, _vp]),
    "carmpc_rollout_bitset_sharded": (_i32, [_vp, _vp, _dp, _dp, _dp, _dp, _i64, _i64, _i64, _vp, _i32, _vp]),
    "carmpc_shard_wait": (_i32, [_vp, _vp, _vp]),
    "carmpc_shard_result": (_i32, [_vp, ctypes.POINTER(_vp), ctypes.POINTER(_i64)]),
    "carmpc_shard_check": (_i32, [_vp]),
    "carmpc_qp_default_opts": (None, [ctypes.POINTER(QPOpts)]),
    "carmpc_qp_create": (_i32, [_i32, _i32, _i32] + [_dp] * 13 + [ctypes.POINTER(QPOpts), ctypes.POINTER(_vp)]),
    "carmpc_qp_get_setup": (_i32, [_vp, _i32, _dp, _i32]),
    "carmpc_qp_solve_batch": (_i32, [_vp, _dp, _dp, _dp, _i64, _dp, _dp, _vp, _vp, _dp, _vp, _i32, _i32, _vp]),
    "carmpc_qp_solve_seeded": (_i32, [_vp, _dp, _dp, _dp, _vp, _i64, _dp, _dp, _vp, _vp, _dp, ctypes.POINTER(_i64), _vp]),
    "carmpc_qp_solve_certified": (_i32, [_vp, _dp, _dp, _dp, _vp, _i64, _dp, _dp, _vp, _vp, _dp, _dp, ctypes.POINTER(_i64),
                                         _vp]),
    "carmpc_qp_sensitivity": (_i32, [_vp, _dp, _dp, _i64, _vp, _dp, _dp, _i32, _dp, _dp, _vp, _vp]),
    "carmpc_qp_checker_create": (_i32, [_i32, _i32] + [_dp] * 9 + [ctypes.POINTER(_vp)]),
    "carmpc_qp_check": (_i32, [_vp, _dp, _dp, _dp, _i64, _vp, _dp, _dp, _dp, _vp]),
    "carmpc_qp_map_host": (_i32, [_vp, _dp, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32),
                                  ctypes.POINTER(ctypes.c_int32), _dp, _dp, _dp, _vp, _vp, ctypes.POINTER(_i64)]),
    "carmpc_qp_solve_host": (_i32, [_vp, _dp, _dp, _dp, _i64, _dp, _dp, _vp, _vp, _dp]),
    "carmpc_qp_polish_stats": (_i32, [_vp, ctypes.POINTER(_i64)]),
    "carmpc_qp_last_stats": (_i32, [_vp, ctypes.POINTER(_i64), ctypes.POINTER(_i64)]),
    "carmpc_qp_tensor_mode": (_i32, [_vp, _i32, ctypes.POINTER(_i64)]),
    "carmpc_closed_loop": (_i32, [_vp, _i32, _dp, _dp, _dp, _dp, _dp, ctypes.c_double, ctypes.c_double, _i32,
                                  _i32, _dp, _dp, _i64, _dp, _vp, _dp, _dp, ctypes.POINTER(_i64), _vp]),
    "carmpc_closed_loop_disturbance": (_i32, [_vp, _dp, _dp, _dp, ctypes.POINTER(DisturbanceModel), _dp, ctypes.c_double,
                                              ctypes.c_double, _i32, _i32, _dp, _dp, _dp, _dp, _i64, _dp, _dp, _vp, _dp,
                                              _dp, _dp, ctypes.POINTER(_i64), _vp]),
    "carmpc_closed_loop_stochastic": (_i32, [_vp, _i32, _dp, _dp, _dp, _dp, ctypes.POINTER(DisturbanceModel), _dp,
                                             ctypes.c_double, ctypes.c_double, _i32, _i32, _dp, _dp, _dp, _dp, _i64, _dp,
                                             _dp, _vp, _dp, _dp, _dp, ctypes.POINTER(LoopNoiseParams), _dp, _i32, _vp, _vp,
                                             _vp, ctypes.POINTER(_i64), _vp]),
    "carmpc_measure_peak": (_i32, [_i32, ctypes.POINTER(ctypes.c_double)]),
}

_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load(rebuild_if_stale: bool = True):
    """Load (building first when the sources are newer) and type every entry point."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if rebuild_if_stale and _build.is_stale():
        try:
            path = _build.build_library()
        except Exception as exc:           # no nvcc on this machine: use what is there, or fail loudly
            if not os.path.isfile(path):
                raise CarmpcError(f"libcarmpc_b200.so is missing and could not be built: {exc}") from exc
    if not os.path.isfile(path):
        raise CarmpcError(f"{path} not found; run `python -m carmpc_b200.build`")
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError here = header / library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().carmpc_last_error().decode(errors="replace")
        raise CarmpcError(f"carmpc error {rc}: {msg}")


def ptr(arr) -> int:
    """Address of a numpy array or torch tensor (None -> NULL)."""
    if arr is None:
        return None
    if hasattr(arr, "data_ptr"):
        return arr.data_ptr()
    return arr.ctypes.data
