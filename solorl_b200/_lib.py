"""Loader of the CUDA C-ABI library ``libsolo_b200.so`` (built in-tree by
``solorl_b200.build.build()`` / ``__graft_entry__.build()``).

There is no CPU fallback: if the library is missing or cannot be loaded this raises,
and ``solo_create`` itself fails with ``SOLO_E_CUDA`` when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

from .abi import SoloEpisodeStats, SoloModelTable, SoloSimParams

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SOLO_B200_LIB", os.path.join(_PKG, "libsolo_b200.so"))   # override: A/B builds
_lib = None

# every symbol include/solo_b200.h declares (tests check the export list against the header)
SYMBOLS = [
    "solo_default_params", "solo_dims", "solo_create", "solo_destroy", "solo_last_error",
    "solo_reset", "solo_step", "solo_step_host", "solo_get_observation", "solo_get_state",
    "solo_set_state", "solo_set_goals", "solo_get_contacts", "solo_get_work_counters", "solo_forward_dynamics",
    "solo_substep", "solo_action_to_torque", "solo_episode_stats", "solo_set_goal_radius",
    "solo_gae", "solo_launch_count", "solo_actuator_step", "solo_get_feet",
    "solo_accumulate_episode_stats", "solo_set_contacts", "solo_step_variant", "solo_set_external_force",
    "solo_get_env_params", "solo_get_push_force",
]


class SoloError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"solo_b200 error {code}: {msg}")
        self.code = code


def lib():
    """Load (once) and return the ctypes library; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build the CUDA extension first "
            "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, fp = C.c_void_p, C.c_void_p  # device pointers are passed as integers
    L.solo_default_params.argtypes = [C.POINTER(SoloSimParams)]
    L.solo_dims.argtypes = [C.POINTER(SoloModelTable), C.POINTER(SoloSimParams)] + [C.POINTER(C.c_int32)] * 4
    L.solo_create.argtypes = [C.POINTER(SoloModelTable), C.POINTER(SoloSimParams), C.c_int32, C.c_int32,
                              C.c_uint64, C.c_int64, C.POINTER(vp)]
    L.solo_destroy.argtypes = [vp]
    L.solo_last_error.argtypes = [vp]
    L.solo_last_error.restype = C.c_char_p
    L.solo_reset.argtypes = [vp, fp, fp, vp]
    L.solo_step.argtypes = [vp, fp, fp, fp, fp, vp]
    L.solo_step_host.argtypes = [vp, fp, fp, fp, fp, vp]
    L.solo_get_observation.argtypes = [vp, fp, vp]
    L.solo_get_state.argtypes = [vp, fp, vp]
    L.solo_set_state.argtypes = [vp, fp, vp]
    L.solo_set_goals.argtypes = [vp, fp, vp]
    L.solo_get_contacts.argtypes = [vp, fp, vp]
    L.solo_set_contacts.argtypes = [vp, fp, vp]
    L.solo_get_work_counters.argtypes = [vp, fp, vp]
    L.solo_forward_dynamics.argtypes = [vp, fp, fp, fp, vp]
    L.solo_substep.argtypes = [vp, fp, vp]
    L.solo_action_to_torque.argtypes = [vp, fp, fp, vp]
    L.solo_get_env_params.argtypes = [vp, fp, vp]
    L.solo_get_push_force.argtypes = [vp, fp, vp]
    L.solo_episode_stats.argtypes = [vp, fp, vp]
    L.solo_actuator_step.argtypes = [vp, fp, C.c_int32, vp]
    L.solo_get_feet.argtypes = [vp, fp, vp]
    L.solo_set_external_force.argtypes = [vp, fp, vp]
    L.solo_accumulate_episode_stats.argtypes = [vp, fp, fp, vp]
    L.solo_set_goal_radius.argtypes = [vp, C.c_double]
    L.solo_gae.argtypes = [fp, fp, fp, fp, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_int32, vp]
    L.solo_launch_count.argtypes = [vp]
    L.solo_launch_count.restype = C.c_int64
    L.solo_step_variant.argtypes = [vp]
    L.solo_step_variant.restype = C.c_char_p
    for name in SYMBOLS:
        if name not in ("solo_last_error", "solo_launch_count", "solo_step_variant"):
            getattr(L, name).restype = C.c_int
    _lib = L
    return L


def check(rc, handle=None):
    if rc != 0:
        msg = lib().solo_last_error(handle)
        raise SoloError(rc, msg.decode() if msg else "?")
