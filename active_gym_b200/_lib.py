"""ctypes binding of ``libagym_b200.so`` (the C ABI declared in ``include/agym_b200.h``).

The product path has NO CPU fallback: if the library is missing or a call fails, a
``RuntimeError`` is raised.  Build it with ``python -m active_gym_b200.build`` (or
``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AGYM_LIB") or os.path.join(_HERE, "lib", "libagym_b200.so")  # AGYM_LIB: timing experiments only

ABI_VERSION = 4

# status codes / flags (mirrors of the header's macros)
OK = 0
FLAG_FRAME_A, FLAG_FRAME_B, FLAG_HARD_RESET, FLAG_IDLE = 1, 2, 4, 8
FOV_APPLY, FOV_RESET, FOV_KEEP = 0, 1, 2
OUT_CROP, OUT_MASK, OUT_RESIZE_FULL, OUT_RESIZE_FOV = 0, 1, 2, 3
ATYPE_FOV_LOC, ATYPE_FOV_RES = 0, 1
ERR_RES_RANGE, ERR_RES_FRACTION = 1, 2
DTYPE_F32, DTYPE_F16, DTYPE_BF16 = 0, 1, 2
BG_ZERO, BG_PERIPHERY = 0, 1

# the symbols include/agym_b200.h declares; tests check that the .so exports every one
EXPORTS = (
    "agym_abi_version", "agym_status_string", "agym_plan_create", "agym_plan_destroy",
    "agym_plan_ring_bytes", "agym_plan_pcache_bytes", "agym_ingest_atari", "agym_ingest_dmc",
    "agym_stack", "agym_observe_fixed", "agym_observe_peripheral", "agym_observe_flexible",
    "agym_synth_frames", "agym_table_cv2", "agym_table_aa", "agym_table_blur", "agym_normalize", "agym_plan_used_rows", "agym_ingest_atari_packed", "agym_record_step",
    "agym_observe_flexible_peripheral", "agym_plan_memory_bytes", "agym_observe_fixed_memory",
    "agym_observe_fixed_memory_paste",
)


class Config(C.Structure):
    """``agym_config`` of the header."""
    _fields_ = [
        ("n_envs", C.c_int32), ("frame_stack", C.c_int32), ("obs_h", C.c_int32), ("obs_w", C.c_int32),
        ("raw_h", C.c_int32), ("raw_w", C.c_int32), ("raw_c", C.c_int32), ("luma_w", C.c_int32 * 3),
        ("fov_h", C.c_int32), ("fov_w", C.c_int32), ("periph_h", C.c_int32), ("periph_w", C.c_int32),
        ("relative", C.c_int32), ("act_lo", C.c_double), ("act_hi", C.c_double), ("fov_init_loc", C.c_double * 2),
        ("no_antialias", C.c_int32), ("obs_c", C.c_int32),
    ]


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built "
            "(run `python -m active_gym_b200.build`); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, i32, u64, sz = C.c_void_p, C.c_int32, C.c_uint64, C.c_size_t
    L.agym_abi_version.restype = C.c_int
    L.agym_status_string.restype = C.c_char_p
    L.agym_status_string.argtypes = [C.c_int]
    L.agym_plan_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.agym_plan_destroy.argtypes = [vp]
    L.agym_plan_ring_bytes.restype = sz
    L.agym_plan_ring_bytes.argtypes = [vp]
    L.agym_plan_pcache_bytes.restype = sz
    L.agym_plan_pcache_bytes.argtypes = [vp]
    L.agym_ingest_atari.argtypes = [vp] * 8
    L.agym_ingest_dmc.argtypes = [vp] * 7
    L.agym_ingest_atari_packed.argtypes = [vp] * 8
    L.agym_plan_used_rows.argtypes = [vp, vp, i32]
    L.agym_stack.argtypes = [vp] * 5
    L.agym_observe_fixed.argtypes = [vp, vp, vp, vp, vp, vp, i32, vp, vp, i32, vp]
    L.agym_observe_peripheral.argtypes = [vp] * 9 + [i32, vp]
    L.agym_observe_flexible.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, i32, vp]
    L.agym_observe_flexible_peripheral.argtypes = [vp] * 12 + [i32, vp]
    L.agym_plan_memory_bytes.restype = sz
    L.agym_plan_memory_bytes.argtypes = [vp, i32]
    L.agym_observe_fixed_memory.argtypes = [vp] * 6 + [i32] + [vp] * 5 + [i32, vp]
    L.agym_observe_fixed_memory_paste.argtypes = [vp] * 7 + [i32, i32] + [vp] * 5 + [i32, vp]
    L.agym_record_step.argtypes = [i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.agym_synth_frames.argtypes = [vp, sz, u64, vp]
    L.agym_normalize.argtypes = [vp, sz, i32, vp, vp]
    L.agym_table_cv2.argtypes = [i32, i32, i32, vp, vp, vp]
    L.agym_table_aa.argtypes = [i32, i32, i32, vp, vp, sz, vp]
    L.agym_table_blur.argtypes = [i32, i32, i32, vp, vp, vp, sz, vp, vp]
    if L.agym_abi_version() != ABI_VERSION:
        raise RuntimeError(f"libagym_b200 ABI {L.agym_abi_version()} != expected {ABI_VERSION}; rebuild")
    _lib = L
    return L


def check(status: int, what: str) -> None:
    if status != OK:
        msg = lib().agym_status_string(status).decode()
        raise RuntimeError(f"{what} failed: {msg} (status {status})")
