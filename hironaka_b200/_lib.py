"""ctypes binding of the C-ABI shared library (include/hironaka_b200.h).

There is NO fallback: if the CUDA library has not been built, every op raises.  Build it with
``python -m hironaka_b200.build`` (or ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes
import os

from . import constants as C

_HERE = os.path.dirname(os.path.abspath(__file__))
# HIRONAKA_B200_LIB points the binding at another build of the same library (tuning variants, tools/)
LIB_PATH = os.environ.get("HIRONAKA_B200_LIB") or os.path.join(_HERE, "_lib", "libhironaka_b200.so")
_lib = None

_p = ctypes.c_void_p
_i32, _i64, _u32, _f32 = ctypes.c_int32, ctypes.c_int64, ctypes.c_uint32, ctypes.c_float

# name -> (restype, argtypes); every symbol declared in include/hironaka_b200.h
SIGNATURES = {
    "hk_version": (ctypes.c_int, []),
    "hk_error_string": (ctypes.c_char_p, [ctypes.c_int]),
    "hk_kernel_class": (ctypes.c_int, [ctypes.c_int, ctypes.c_int]),
    "hk_debug_force_generic": (ctypes.c_int, [ctypes.c_int]),
    "hk_debug_set_pdl": (ctypes.c_int, [ctypes.c_int]),
    "hk_step": (ctypes.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _u32, _u32, _f32, _f32, _p]),
    "hk_step_census": (ctypes.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _u32, _u32, _f32, _f32, _p]),
    "hk_step_census_obs": (ctypes.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _u32, _u32, _f32,
                                          _f32, _p]),
    "hk_census_bytes": (_i64, [_i64, _i32, _i32]),
    "hk_debug_set_session_graphs": (ctypes.c_int, [ctypes.c_int]),
    "hk_shift": (ctypes.c_int, [_p, _p, _p, _p, _i64, _i32, _i32, _i32, _u32, _f32, _p]),
    "hk_reposition": (ctypes.c_int, [_p, _p, _i64, _i32, _i32, _i32, _f32, _p]),
    "hk_newton_polytope": (ctypes.c_int, [_p, _p, _i64, _i32, _i32, _i32, _f32, _p]),
    "hk_rescale": (ctypes.c_int, [_p, _p, _i64, _i32, _i32, _i32, _f32, _p]),
    "hk_features": (ctypes.c_int, [_p, _p, _p, _i64, _i32, _i32, _i32, _u32, _f32, _p]),
    "hk_dones": (ctypes.c_int, [_p, _p, _p, _i64, _i32, _i32, _i32, _p]),
    "hk_host_policy": (ctypes.c_int, [_p, _p, _i64, _i32, _i32, _i32, _u32, _f32, _p]),
    "hk_rollout": (ctypes.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _u32, _u32, _f32, _p]),
    "hk_rollout_seeded": (ctypes.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _u32, _u32, _f32,
                                         ctypes.c_uint64, _i32, _p]),
    "hk_random_actions": (ctypes.c_int, [_p, _p, _i64, _i32, _i32, ctypes.c_uint64, _i32, _p]),
    "hk_rollout_record": (ctypes.c_int, [_p, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _u32,
                                         _u32, _f32, ctypes.c_uint64, _i32, _p]),
    "hk_rollout_threshold": (ctypes.c_int, [_p, _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _i32,
                                            _u32, _u32, _f32, ctypes.c_uint64, _i32, _f32, _i32, _p, _p]),
    "hk_search_workspace_bytes": (_i64, [_i64, _i32, _i32, _i64]),
    "hk_search_depth": (ctypes.c_int, [_p, _p, _p, _p, _i64, _i32, _i32, _i32, _u32, _u32, _i32, _i64, _i64, _p, _p]),
    "hk_search_value_workspace_bytes": (_i64, [_i64, _i32, _i32, _i64, _i64]),
    "hk_search_value": (ctypes.c_int, [_p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _u32, _i32, _i64, _i64, _i64, _p, _p]),
    "hk_search_depth_line_workspace_bytes": (_i64, [_i64, _i32, _i32, _i64, _i64]),
    "hk_search_depth_line": (ctypes.c_int, [_p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _u32, _u32, _i32, _i64, _i64, _i64,
                                            _p, _p]),
    "hk_search_value_line": (ctypes.c_int, [_p, _p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _u32, _i32, _i64, _i64, _i64,
                                            _p, _p]),
    "hk_search_value_labels_workspace_bytes": (_i64, [_i64, _i32, _i32, _i64, _i64]),
    "hk_search_value_labels": (ctypes.c_int, [_p, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _i32,
                                              _u32, _i32, _i64, _i64, _i64, _p, _p]),
    "hk_experience_scratch_words": (_i64, [_i64]),
    "hk_experience_append": (ctypes.c_int, [_p, _p, _p, _i32, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p, _p,
                                            _p, _p, _i64, _p]),
    "hk_value_targets": (ctypes.c_int, [_p, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _f32, _i32, _i32, _i32, _p]),
    "hk_overflow": (ctypes.c_int, [_p, _p, _i64, _i32, _i32, _i32, _f32, _i32, _p]),
    "hk_pack_coords": (ctypes.c_int, [_p, _i32, _p, _i64, _i32, _p]),
    "hk_session_create": (ctypes.c_int, [ctypes.POINTER(_p), ctypes.c_int, _i64, _i32, _i32, _i32, _f32]),
    "hk_session_destroy": (ctypes.c_int, [_p]),
    "hk_session_set_state": (ctypes.c_int, [_p, _p]),
    "hk_session_get_state": (ctypes.c_int, [_p, _p]),
    "hk_session_step": (ctypes.c_int, [_p, _p, _p, _p, _p, _p, _u32, _u32]),
    "hk_session_rollout": (ctypes.c_int, [_p, _p, _p, _i32, _p, _u32, _u32]),
    "hk_session_rollout_ex": (ctypes.c_int, [_p, _p, _p, _i32, _p, _p, _u32, _u32]),
    "hk_session_rollout_bits": (ctypes.c_int, [_p, _p, _p, _i32, _p, _p, _u32, _u32]),
    "hk_session_state_ptr": (_p, [_p]),
    "hk_session_stream": (_p, [_p]),
}


class HironakaB200Error(RuntimeError):
    pass


def lib():
    """The loaded library; raises if it was not built (no CPU or torch fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HironakaB200Error(
                f"{LIB_PATH} is missing: the CUDA extension has not been built. "
                "Run `python -m hironaka_b200.build` (needs nvcc). There is no fallback path.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        v = L.hk_version()
        if v != C.HK_VERSION:
            raise HironakaB200Error(f"library version {v} != python binding version {C.HK_VERSION}; rebuild")
        _lib = L
    return _lib


def check(rc: int, what: str = "hk call") -> None:
    if rc != 0:
        msg = lib().hk_error_string(rc).decode()
        raise HironakaB200Error(f"{what} failed with code {rc}: {msg}")
