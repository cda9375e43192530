"""ctypes binding of libdpomp.so (include/dpomp.h).  This is the only way the host code reaches the GPU.

There is NO CPU fallback: if the shared library is missing, or no CUDA device is present when a compute entry point
is called, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

MAX_COMPARTMENTS = 8
MAX_EVENTS = 8
MAX_PARAMS = 16
MAX_OBS_VALS = 8

RS_SYSTEMATIC, RS_STRATIFIED, RS_MULTINOMIAL = 1, 2, 3
SIM_F32, SIM_F64 = 0, 1
SCATTER_REFERENCE, SCATTER_INTERLEAVED = 0, 1
OBS_GAUSSIAN, OBS_POISSON, OBS_BINOMIAL, OBS_NEGBIN = 0, 1, 2, 3

_HERE = os.path.dirname(os.path.abspath(__file__))
# DPOMP_LIB_PATH selects another build of the same library (kernel A/B measurements); there is still no fallback
LIB_PATH = os.environ.get("DPOMP_LIB_PATH") or os.path.join(_HERE, "lib", "libdpomp.so")


class DpompError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libdpomp error {code}: {msg}")
        self.code = code


class ModelDesc(C.Structure):
    """struct dpomp_model_desc (include/dpomp.h) -- field order is ABI."""

    _fields_ = [
        ("n_compartments", C.c_int32),
        ("n_events", C.c_int32),
        ("n_params", C.c_int32),
        ("t0_index", C.c_int32),
        ("rate_par", C.c_int32 * MAX_EVENTS),
        ("rate_f1", (C.c_int32 * MAX_COMPARTMENTS) * MAX_EVENTS),
        ("rate_k1", C.c_int32 * MAX_EVENTS),
        ("rate_f2", (C.c_int32 * MAX_COMPARTMENTS) * MAX_EVENTS),
        ("rate_k2", C.c_int32 * MAX_EVENTS),
        ("rate_has_den", C.c_int32 * MAX_EVENTS),
        ("rate_dn", (C.c_int32 * MAX_COMPARTMENTS) * MAX_EVENTS),
        ("rate_kd", C.c_int32 * MAX_EVENTS),
        ("trans", (C.c_int32 * MAX_COMPARTMENTS) * MAX_EVENTS),
        ("initial_condition", C.c_int64 * MAX_COMPARTMENTS),
        ("obs_sigma", C.c_double),
        ("obs_xmask", C.c_int32 * MAX_COMPARTMENTS),
        ("n_obs_vals", C.c_int32),
        ("obs_ymask", C.c_int32 * MAX_OBS_VALS),
        ("n_obs", C.c_int32),
        ("obs_time", C.POINTER(C.c_double)),
        ("obs_id", C.POINTER(C.c_int32)),
        ("obs_val", C.POINTER(C.c_int64)),
    ]


_lib: Optional[C.CDLL] = None

_P = C.c_void_p
_SIGS = {
    "dpomp_last_error": (C.c_char_p, []),
    "dpomp_version": (C.c_int, []),
    "dpomp_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "dpomp_model_create": (C.c_int, [C.POINTER(ModelDesc), C.POINTER(_P)]),
    "dpomp_model_destroy": (C.c_int, [_P]),
    "dpomp_model_set_obs_model": (C.c_int, [_P, C.c_int32, _P, _P]),
    "dpomp_pf_create": (C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, C.c_uint64, C.c_int32, C.POINTER(_P)]),
    "dpomp_pf_destroy": (C.c_int, [_P]),
    "dpomp_pf_set_sim_precision": (C.c_int, [_P, C.c_int32]),
    "dpomp_pf_set_max_events": (C.c_int, [_P, C.c_int64]),
    "dpomp_pf_set_batch_offset": (C.c_int, [_P, C.c_int64]),
    "dpomp_pf_set_fused": (C.c_int, [_P, C.c_int32]),
    "dpomp_pf_set_persistent": (C.c_int, [_P, C.c_int32]),
    "dpomp_pf_set_scatter": (C.c_int, [_P, C.c_int32]),
    "dpomp_pf_set_filter_ids": (C.c_int, [_P, _P, C.c_int32]),
    "dpomp_pf_set_stream_key": (C.c_int, [_P, C.c_uint64]),
    "dpomp_pf_get_stream_key": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "dpomp_pf_geometry": (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "dpomp_pf_loglik": (C.c_int, [_P, _P, C.c_int32, _P]),
    "dpomp_pf_partial": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, _P]),
    "dpomp_pf_permute": (C.c_int, [_P, _P, C.c_int32]),
    "dpomp_pf_copy_filters": (C.c_int, [_P, _P, _P, _P, C.c_int32]),
    "dpomp_pf_get_pop": (C.c_int, [_P, C.c_int32, _P]),
    "dpomp_pf_set_pop": (C.c_int, [_P, C.c_int32, _P]),
    "dpomp_pf_get_last_logw": (C.c_int, [_P, C.c_int32, _P]),
    "dpomp_pf_get_last_ancestors": (C.c_int, [_P, C.c_int32, _P]),
    "dpomp_pf_set_record_ancestors": (C.c_int, [_P, C.c_int32]),
    "dpomp_pf_overflow_count": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "dpomp_pf_last_event_count": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "dpomp_pf_last_timing": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_int32)]),
    "dpomp_pf_set_kernel_timing": (C.c_int, [_P, C.c_int32]),
    "dpomp_pf_last_kernel_timing": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_int32)]),
    "dpomp_pf_export_filters": (C.c_int, [_P, _P, C.c_int32, _P]),
    "dpomp_pf_import_filters": (C.c_int, [_P, _P, C.c_int32, _P]),
    "dpomp_pf_loglik_device": (C.c_int, [_P, _P, C.c_int32, _P]),
    "dpomp_mbp_create": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_uint64, C.c_int32, C.POINTER(_P)]),
    "dpomp_mbp_destroy": (C.c_int, [_P]),
    "dpomp_mbp_set_batch_offset": (C.c_int, [_P, C.c_int64]),
    "dpomp_mbp_set_stream_key": (C.c_int, [_P, C.c_uint64]),
    "dpomp_mbp_set_mode": (C.c_int, [_P, C.c_int32]),
    "dpomp_mbp_reset": (C.c_int, [_P]),
    "dpomp_mbp_iterate": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, _P]),
    "dpomp_mbp_propose": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, _P]),
    "dpomp_mbp_accept": (C.c_int, [_P, _P, C.c_int32]),
    "dpomp_mbp_permute": (C.c_int, [_P, _P, C.c_int32]),
    "dpomp_mbp_get_lengths": (C.c_int, [_P, _P, C.c_int32, _P]),
    "dpomp_mbp_export": (C.c_int, [_P, _P, _P, C.c_int32, _P, _P, _P]),
    "dpomp_mbp_import": (C.c_int, [_P, _P, _P, C.c_int32, _P, _P, _P]),
    "dpomp_mbp_outer_begin": (C.c_int, [_P, _P, C.c_int64, _P, _P, _P]),
    "dpomp_mbp_outer_iterate": (C.c_int, [_P, C.c_int32, C.c_int32, _P]),
    "dpomp_mbp_outer_moments": (C.c_int, [_P, _P, _P]),
    "dpomp_mbp_outer_resample": (C.c_int, [_P, C.c_int32, _P, C.c_int64, _P]),
    "dpomp_mbp_outer_sweep": (C.c_int, [_P, _P, _P, C.c_double, C.c_int32, C.c_int32, _P]),
    "dpomp_mbp_outer_get": (C.c_int, [_P, _P, _P]),
    "dpomp_mbp_outer_end": (C.c_int, [_P]),
    "dpomp_mbp_capacity": (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "dpomp_mbp_reserve": (C.c_int, [_P, C.c_int32]),
    "dpomp_mbp_get_states": (C.c_int, [_P, C.c_int32, _P]),
    "dpomp_mbp_get_particle": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P, C.c_int64, _P]),
    "dpomp_comm_unique_id": (C.c_int, [_P, C.c_int32]),
    "dpomp_comm_create": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "dpomp_comm_destroy": (C.c_int, [_P]),
    "dpomp_comm_info": (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "dpomp_comm_barrier": (C.c_int, [_P]),
    "dpomp_partition_bounds": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dpomp_comm_allgather_f64": (C.c_int, [_P, _P, C.c_int64, C.c_int32, _P]),
    "dpomp_pf_partial_allgather": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int64, _P]),
    "dpomp_pf_resample_migrate": (C.c_int, [_P, _P, _P, C.c_int64]),
    "dpomp_mbp_resample_migrate": (C.c_int, [_P, _P, _P, C.c_int64]),
    "dpomp_debug_uniforms_f32": (C.c_int, [_P, C.c_int32, _P, _P]),
    "dpomp_resample_indices": (
        C.c_int,
        [C.c_int32, C.c_int32, _P, C.c_int64, _P, C.c_int64, C.c_int64, _P, C.c_int32],
    ),
}

EXPORTED_SYMBOLS = tuple(_SIGS.keys())


def lib() -> C.CDLL:
    """Load libdpomp.so (built in-tree by `__graft_entry__.build()` / discretepomp.jl_b200/build.py)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build the CUDA extension first (python __graft_entry__.py build). "
                "There is no CPU fallback for the particle-filter path."
            )
        handle = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        lenient = os.environ.get("DPOMP_LIB_LENIENT") == "1"  # A/B of OLDER builds only (scripts/ab_commits.sh)
        for name, (res, args) in _SIGS.items():
            if lenient and not hasattr(handle, name):
                continue
            fn = getattr(handle, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(code: int) -> None:
    if code != 0:
        msg = lib().dpomp_last_error()
        raise DpompError(code, msg.decode() if msg else "unknown")


def ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def as_f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def as_i64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.int64)
