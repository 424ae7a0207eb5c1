"""Loader + ctypes prototypes of libdrloco_b200.so (the CUDA library; built in-tree by __graft_entry__.build()).

There is no CPU fallback: if the shared library is missing or cannot be loaded this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

from .cabi import DrlConfig, DrlWalkerModel, DRL_ABI_VERSION

_HERE = os.path.dirname(os.path.abspath(__file__))
# developer hook: DRLOCO_B200_LIB points at another build of the same ABI (A/B runs of kernel variants); default in-tree
LIB_PATH = os.environ.get("DRLOCO_B200_LIB") or os.path.join(_HERE, "libdrloco_b200.so")
_LIB = None

vp, i32, f32 = C.c_void_p, C.c_int32, C.c_float

# name -> (restype, argtypes); mirrors include/drloco_b200.h one to one
PROTOTYPES = {
    "drl_version": (C.c_int, []),
    "drl_last_error": (C.c_char_p, []),
    "drl_create": (C.c_int, [C.POINTER(DrlConfig), C.POINTER(vp)]),
    "drl_destroy": (C.c_int, [vp]),
    "drl_upload_model": (C.c_int, [vp, C.POINTER(DrlWalkerModel)]),
    "drl_upload_mocap": (C.c_int, [vp, i32, i32, vp, i32, vp, vp, vp, vp, vp, i32, i32, vp, i32]),
    "drl_reset": (C.c_int, [vp, vp, vp, vp, vp, vp]),
    "drl_step": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "drl_get_state": (C.c_int, [vp, vp, vp, vp, vp]),
    "drl_set_state": (C.c_int, [vp, vp, vp, vp, vp]),
    "drl_get_extras": (C.c_int, [vp, vp, vp]),
    "drl_get_stats": (C.c_int, [vp, vp, vp]),
    "drl_reset_stats": (C.c_int, [vp, vp]),
    "drl_get_episode_ring": (C.c_int, [vp, vp, vp, i32, C.POINTER(C.c_int64), vp]),
    "drl_get_episode_positions": (C.c_int, [vp, vp, vp, vp, i32, vp]),
    "drl_get_running_rsi_positions": (C.c_int, [vp, vp, vp]),
    "drl_get_median_torque": (C.c_int, [vp, vp, vp]),
    "drl_get_ee_reward": (C.c_int, [vp, vp, vp, vp]),
    "drl_set_eval_mode": (C.c_int, [vp, i32]),
    "drl_set_det_init_counters": (C.c_int, [vp, vp]),
    "drl_set_speed_profile": (C.c_int, [vp, vp, i32]),
    "drl_set_seed": (C.c_int, [vp, C.c_uint64]),
    "drl_set_playback": (C.c_int, [vp, i32]),
    "drl_set_ref_obs": (C.c_int, [vp, i32, vp]),
    "drl_set_actuation": (C.c_int, [vp, i32, vp, vp]),
    "drl_set_contact_termination": (C.c_int, [vp, C.c_uint32]),
    "drl_get_contact_terminations": (C.c_int, [vp, vp, vp]),
    "drl_set_adaptive_rsi": (C.c_int, [vp, f32, i32, i32]),
    "drl_get_adaptive_rsi": (C.c_int, [vp, vp, vp, vp, vp, vp]),
    "drl_set_adaptive_rsi_counts": (C.c_int, [vp, vp, vp]),
    "drl_set_mocap_clips": (C.c_int, [vp, i32, vp, vp]),
    "drl_get_clip_stats": (C.c_int, [vp, vp, vp]),
    "drl_launch_info": (C.c_int, [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]),
    "drl_debug_set": (C.c_int, [vp, i32, i32, i32]),
    "drl_debug_read": (C.c_int, [vp, vp, i32]),
    "drl_attach_vecnorm": (C.c_int, [vp, vp, f32, vp]),
    "drl_comm_create": (C.c_int, [i32, i32, i32, C.POINTER(vp)]),
    "drl_comm_export": (C.c_int, [vp, vp]),
    "drl_comm_connect": (C.c_int, [vp, vp]),
    "drl_comm_destroy": (C.c_int, [vp]),
    "drl_vecnorm_step": (C.c_int, [vp, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, f32, f32, f32, i32, vp, i32, vp]),
    "drl_vecnorm_terminal_compact": (C.c_int, [vp, vp, i32, i32, vp, f32, f32, i32, vp, vp, vp]),
    "drl_fp32_peak_probe": (C.c_int, [i32, C.POINTER(C.c_double)]),
    "drl_vecnorm_moments": (C.c_int, [vp, i32, i32, vp, vp, f32, vp, vp]),
}


class DrlError(RuntimeError):
    pass


def load():
    """dlopen the CUDA library; raises if it has not been built (no fallback path exists)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise DrlError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(nvcc, sm_100a). drloco_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if the library does not export the symbol
        fn.restype, fn.argtypes = res, args
    if lib.drl_version() != DRL_ABI_VERSION:
        raise DrlError(f"ABI mismatch: library {lib.drl_version()} vs python {DRL_ABI_VERSION}")
    _LIB = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().drl_last_error().decode("utf-8", "replace")
        raise DrlError(f"{what} failed ({rc}): {msg}")
