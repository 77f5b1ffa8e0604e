"""ctypes binding of librbm_b200.so -- the C ABI declared in include/rbm_b200.h.

There is no CPU fallback anywhere in this package: if the shared library cannot be loaded (and cannot be
built because nvcc is absent) importing the compute layer raises; if it loads but no CUDA device is
present every compute entry point returns RBM_ERR_CUDA, surfaced here as `RbmCudaError`.
"""
from __future__ import annotations

import ctypes as C
import os
import re
import threading

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "librbm_b200.so")
HEADER = os.path.join(os.path.dirname(_PKG), "include", "rbm_b200.h")

RBM_OK, RBM_ERR_INVALID, RBM_ERR_CUDA, RBM_ERR_UNSUPPORTED, RBM_ERR_NCCL = 0, -1, -2, -3, -4
FLAG_FORCE_GENERIC = 1
FLAG_NO_TMA = 2
PATH_NAMES = {0: "generic", 1: "seq_iso", 2: "seq_rigid"}


class RbmError(RuntimeError):
    pass


class RbmCudaError(RbmError):
    pass


class RbmNcclError(RbmError):
    pass


_lock = threading.Lock()
_lib = None

_dp = C.POINTER(C.c_double)
_vp = C.c_void_p
_i64 = C.c_int64

# name -> (restype, argtypes).  tests/test_abi.py checks this table against the header.
SIGNATURES = {
    "rbm_version": (C.c_char_p, []),
    "rbm_last_error_string": (C.c_char_p, []),
    "rbm_device_count": (C.c_int, []),
    "rbm_device_pci_bus_id": (C.c_int, [C.c_int, C.c_char_p, C.c_int]),
    "rbm_model_create": (C.c_int, [C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_uint, C.c_int, C.POINTER(_vp)]),
    "rbm_model_destroy": (None, [_vp]),
    "rbm_model_analyze": (C.c_int, [C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_uint, C.POINTER(C.c_int), _vp, _vp]),
    "rbm_fast_param_count": (C.c_int, []),
    "rbm_generic_param_count": (C.c_int, [C.c_int]),
    "rbm_model_num_joints": (C.c_int, [_vp]),
    "rbm_model_kernel_path": (C.c_int, [_vp]),
    "rbm_rnea_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "rbm_rnea_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "rbm_rnea_aos_f64": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "rbm_rnea_aos_f32": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "rbm_rnea_full_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "rbm_rnea_full_host_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64]),
    "rbm_rnea_planned_f64": (C.c_int, [_vp, _vp, _vp, _vp, C.c_double, C.c_double, C.c_double, _vp, _vp, _i64, _i64, _vp]),
    "rbm_rnea_planned_f32": (C.c_int, [_vp, _vp, _vp, _vp, C.c_double, C.c_double, C.c_double, _vp, _vp, _i64, _i64, _vp]),
    "rbm_rnea_host_f64": (C.c_int, [_vp, _vp, _vp, _i64, _i64]),
    "rbm_rnea_host_f32": (C.c_int, [_vp, _vp, _vp, _i64, _i64]),
    "rbm_model_live_inputs": (C.c_int, [_vp, _vp]),
    "rbm_rnea_host_soa_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64]),
    "rbm_rnea_host_soa_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64]),
    "rbm_rnea_planned_host_f64": (C.c_int, [_vp, _vp, _vp, _vp, C.c_double, C.c_double, C.c_double, _vp, _i64, _i64, _i64]),
    "rbm_rnea_planned_host_f32": (C.c_int, [_vp, _vp, _vp, _vp, C.c_double, C.c_double, C.c_double, _vp, _i64, _i64, _i64]),
    "rbm_regressor_rows_f64": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "rbm_sensor_twists_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "rbm_regressor_from_traj_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "rbm_regressor_from_traj_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "rbm_gram_workspace_bytes": (C.c_size_t, [_vp, _i64]),
    "rbm_regressor_gram_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_size_t, _i64, _i64, _vp]),
    "rbm_regressor_gram_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_size_t, _i64, _i64, _vp]),
    "rbm_payload_regressor_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "rbm_payload_regressor_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "rbm_payload_gram_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_size_t, _i64, _i64, _vp]),
    "rbm_payload_gram_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_size_t, _i64, _i64, _vp]),
    "rbm_nccl_available": (C.c_int, []),
    "rbm_nccl_unique_id": (C.c_int, [_vp]),
    "rbm_nccl_comm_create": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "rbm_nccl_comm_destroy": (C.c_int, [_vp]),
    "rbm_allreduce_gram": (C.c_int, [_vp, _vp, _vp]),
    "rbm_allreduce_gram_n": (C.c_int, [_vp, _vp, _i64, _vp]),
    "rbm_linearize_f64": (C.c_int, [_vp, _vp, _vp, _vp, C.c_double, C.c_double, C.c_int, _vp, _vp, _vp, _i64, _i64, _vp]),
    "rbm_forward_dynamics_f64": (C.c_int, [_vp, _vp, _vp, _vp, C.c_double, _vp, _vp, _vp, _i64, _i64, _vp]),
    "rbm_regressor_gram_grouped_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _i64, _i64, _i64, _vp]),
    "rbm_closed_loop_f64": (C.c_int, [_vp, _vp, _vp, _vp, C.c_double, C.c_double, _i64, _vp, _vp, C.c_double, C.c_double, C.c_double, _vp, _vp, _vp, _i64,
                                      _vp, _vp, _vp, _i64, _i64, _vp]),
    "rbm_transfer_simat_f64": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "rbm_coordinate_transfer_simat_f64": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "rbm_coordinate_transfer_imat_f64": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _vp]),
    "rbm_spatial_inertia_f64": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "rbm_compose_f64": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _i64, _vp]),
    "rbm_point_motion_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _vp]),
}


def header_symbols():
    """Every function name declared with RBM_API in include/rbm_b200.h."""
    with open(HEADER) as f:
        text = f.read()
    return re.findall(r"RBM_API\s+[\w\s\*]+?\b(rbm_\w+)\s*\(", text)


def load():
    """Load and type the library.  The in-tree build is refreshed first whenever it is missing or STALE: `build_library()` compares a
    fingerprint of csrc/ + the header + the flags with the one recorded at the last build and returns at once when they match, so
    an edited kernel can never run as an old binary.  Without nvcc a stale or missing library is an error (no fallback)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        from . import build as _build

        if _build.have_nvcc():
            _build.build_library(force=bool(os.environ.get("RBM_REBUILD")))
        elif not os.path.exists(LIB_PATH):
            raise RbmError(f"{LIB_PATH} is missing and nvcc is not available to build it")
        elif not _build.is_fresh():
            raise RbmError(f"{LIB_PATH} is stale (csrc/ changed since it was built) and nvcc is not available to rebuild it")
        try:
            lib = C.CDLL(LIB_PATH)
        except OSError as e:  # no silent fallback
            raise RbmError(f"cannot load {LIB_PATH}: {e}. Build it with `python -m rigid_body_manipulation_b200.build`.") from e
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def last_error() -> str:
    return load().rbm_last_error_string().decode()


def check(rc: int, what: str = ""):
    if rc == RBM_OK:
        return
    msg = f"{what}: {last_error()}" if what else last_error()
    if rc == RBM_ERR_INVALID:
        raise ValueError(msg)
    if rc == RBM_ERR_CUDA:
        raise RbmCudaError(msg)
    if rc == RBM_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == RBM_ERR_NCCL:
        raise RbmNcclError(msg)
    raise RbmError(f"{msg} (status {rc})")
