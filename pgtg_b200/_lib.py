"""ctypes binding of the C ABI (include/pgtg_b200.h).

`load()` opens the in-tree CUDA library pgtg_b200/libpgtg_b200.so. There is no fallback: if the
library has not been built (python -c "import __graft_entry__ as g; g.build()") this raises.
"""
from __future__ import annotations

import ctypes as C
import os

from .config import PgtgConfig, PgtgRule, PgtgTile

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpgtg_b200.so")

OBS_FORMATS = {"int8": 0, "bits": 1}  # PGTG_OBS_INT8 / PGTG_OBS_BITS
UNPACK_FORMATS = {"int8": 0, "flat": 1}  # PGTG_UNPACK_INT8 / PGTG_UNPACK_FLAT

STATE_FIELDS = ("agent", "flat_tire", "light_counter", "elapsed", "num_cars", "cars", "tiles", "plan", "used",
                "draw_cursor", "error")


class PgtgState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in STATE_FIELDS]


class PgtgBuffers(C.Structure):
    _fields_ = [("num_envs", C.c_int32), ("num_channels", C.c_int32), ("window", C.c_int32), ("max_cars", C.c_int32)] + [
        (n, C.c_void_p) for n in (
            "obs_map", "obs_position", "obs_velocity", "obs_next_subgoal_direction", "reward", "cost", "terminated",
            "truncated", "step_state", "step_flags", "final_obs_map", "final_obs_position", "final_obs_velocity",
            "final_obs_next_subgoal_direction", "stats")]


EXPORTS = {
    "pgtg_last_error": (C.c_char_p, []),
    "pgtg_abi_version": (C.c_int, []),
    "pgtg_create": (C.c_int, [C.POINTER(PgtgConfig), C.c_int, C.POINTER(C.c_void_p)]),
    "pgtg_destroy": (C.c_int, [C.c_void_p]),
    "pgtg_load_fixed_map": (C.c_int, [C.c_void_p, C.POINTER(PgtgTile)] + [C.c_int] * 8),
    "pgtg_load_direction_lut": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "pgtg_load_draws": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pgtg_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pgtg_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "pgtg_step_host": (C.c_int, [C.c_void_p] * 9),
    "pgtg_packed_obs_bytes": (C.c_int64, [C.c_void_p]),
    "pgtg_step_host_packed": (C.c_int, [C.c_void_p] * 8 + [C.c_int, C.c_void_p]),
    "pgtg_host_sync": (C.c_int, [C.c_void_p]),
    "pgtg_unpack_obs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int]),
    "pgtg_state_bytes": (C.c_int64, [C.c_void_p]),
    "pgtg_save_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "pgtg_load_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "pgtg_copy_state": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pgtg_set_evaluation": (C.c_int, [C.c_void_p, C.c_double, C.c_int]),
    "pgtg_observe": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pgtg_update_rules": (C.c_int, [C.c_void_p, C.POINTER(PgtgRule), C.c_int]),
    "pgtg_get_buffers": (C.c_int, [C.c_void_p, C.POINTER(PgtgBuffers)]),
    "pgtg_dlpack": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]),
    "pgtg_get_state": (C.c_int, [C.c_void_p, C.POINTER(PgtgState)]),
    "pgtg_set_state": (C.c_int, [C.c_void_p, C.POINTER(PgtgState)]),
    "pgtg_get_info": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pgtg_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "pgtg_reduce_stats": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pgtg_reset_stats": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pgtg_launch_count": (C.c_int64, [C.c_void_p]),
    "pgtg_error_summary": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32)]),
    "pgtg_kernel_info": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "pgtg_flatten": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int)]),
    "pgtg_enable_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "pgtg_set_overlap": (C.c_int, [C.c_void_p, C.c_int]),
    "pgtg_levels": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "pgtg_set_obs_format": (C.c_int, [C.c_void_p, C.c_int]),
    "pgtg_expand_obs": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "pgtg_unpack_bits": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int] + [C.c_void_p] * 6),
    "pgtg_timing": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]),
}

_cache: dict[str, C.CDLL] = {}


def load(path: str | None = None) -> C.CDLL:
    path = path or os.environ.get("PGTG_B200_LIB") or LIB_PATH  # env override: A/B builds of the same CUDA library
    if path in _cache:
        return _cache[path]
    if not os.path.exists(path):
        raise RuntimeError(
            f"pgtg_b200: native library {path} is missing. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export the declared ABI
        fn.restype, fn.argtypes = res, args
    if lib.pgtg_abi_version() != 2:
        raise RuntimeError("pgtg_b200: ABI version mismatch between the Python host and the native library")
    _cache[path] = lib
    return lib


def check(lib, rc: int):
    if rc == 0:
        return
    msg = (lib.pgtg_last_error() or b"").decode()
    if rc == -1:
        raise ValueError(msg)
    raise RuntimeError(msg)
