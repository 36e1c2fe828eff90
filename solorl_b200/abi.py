"""ctypes mirrors of the structs in ``include/solo_b200.h`` and the mapping from a
reference YAML config (``configs/*.yaml``; keys read at ``baseEnv.py:8-16``) onto
``SoloSimParams``."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from .model import SoloModel

ABI_VERSION = 3
MAX_LINKS = 20
MAX_FEET = 4

CONTROL_TORQUE, CONTROL_PD, CONTROL_VPD = 0, 1, 2
TASK_STAND, TASK_WALK, TASK_POINTGOAL = 0, 1, 2
RESET_CACHED, RESET_SIMULATE = 0, 1

_CONTROL_NAMES = {  # solo.py:228,231,242
    "torque": CONTROL_TORQUE,
    "pd": CONTROL_PD, "fpd": CONTROL_PD, "fixed_pd": CONTROL_PD,
    "vpd": CONTROL_VPD, "variable_pd": CONTROL_VPD,
}
_TASK_NAMES = {"stand": TASK_STAND, "walk": TASK_WALK, "pointgoal": TASK_POINTGOAL}


class SoloModelTable(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("num_links", C.c_int32),
        ("parent", C.c_int32 * MAX_LINKS),
        ("jtype", C.c_int32 * MAX_LINKS),
        ("axis", (C.c_double * 3) * MAX_LINKS),
        ("origin", (C.c_double * 3) * MAX_LINKS),
        ("mass", C.c_double * MAX_LINKS),
        ("com", (C.c_double * 3) * MAX_LINKS),
        ("inertia", (C.c_double * 6) * MAX_LINKS),
        ("base_mass", C.c_double),
        ("base_com", C.c_double * 3),
        ("base_inertia", C.c_double * 6),
        ("num_feet", C.c_int32),
        ("foot_link", C.c_int32 * MAX_FEET),
        ("foot_center", (C.c_double * 3) * MAX_FEET),
        ("foot_radius", C.c_double),
    ]


class SoloSimParams(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("dt", C.c_double),
        ("frame_skip", C.c_int32),
        ("gravity_z", C.c_double),
        ("lin_damping", C.c_double),
        ("ang_damping", C.c_double),
        ("max_coord_vel", C.c_double),
        ("solver_iters", C.c_int32),
        ("solver_residual_threshold", C.c_double),
        ("contact_erp", C.c_double),
        ("contact_slop", C.c_double),
        ("contact_margin", C.c_double),
        ("friction", C.c_double),
        ("cone_friction", C.c_int32),
        ("torque_hold", C.c_int32),
        ("control", C.c_int32),
        ("kp", C.c_double),
        ("kd", C.c_double),
        ("max_torque", C.c_double),
        ("joint_state_limit", C.c_double),
        ("joint_vel_limit", C.c_double),
        ("task", C.c_int32),
        ("episode_length", C.c_int32),
        ("num_history_stack", C.c_int32),
        ("initial_z", C.c_double),
        ("settle_min", C.c_int32),
        ("settle_max", C.c_int32),
        ("goal_radius", C.c_double),
        ("goal_reach_dist", C.c_double),
        ("pointgoal_dt", C.c_double),
        ("contact_flag_force", C.c_double),
        ("fall_z", C.c_double),
        ("stand_z", C.c_double),
        ("reset_mode", C.c_int32),
        ("joint_limits", C.c_int32),
        ("limit_rows_per_leg", C.c_int32),
        ("joint_limit_erp", C.c_double),
        ("joint_limit_max_impulse", C.c_double),
        ("split_impulse_threshold", C.c_double),
        ("body_contacts", C.c_int32),
        ("knee_radius", C.c_double),
        ("base_half_x", C.c_double),
        ("base_half_y", C.c_double),
        ("base_z_lo", C.c_double),
        ("base_z_hi", C.c_double),
        ("randomize", C.c_int32),
        ("friction_lo", C.c_double),
        ("friction_hi", C.c_double),
        ("base_mass_scale_lo", C.c_double),
        ("base_mass_scale_hi", C.c_double),
        ("motor_strength_lo", C.c_double),
        ("motor_strength_hi", C.c_double),
        ("push_force", C.c_double),
        ("push_interval", C.c_int32),
        ("push_duration", C.c_int32),
    ]


class SoloEpisodeStats(C.Structure):
    _fields_ = [
        ("episode_reward", C.c_float),
        ("episode_return", C.c_float),
        ("episode_length", C.c_int32),
        ("success", C.c_int32),
        ("timeout", C.c_int32),
        ("goals_reached", C.c_int32),
        ("dr_stand", C.c_float),
        ("dr_joint_pose", C.c_float),
        ("dr_torque", C.c_float),
        ("dr_balance", C.c_float),
        ("dr_progress", C.c_float),
        ("nan", C.c_int32),
    ]


EPISODE_STATS_DTYPE = np.dtype([
    ("episode_reward", np.float32), ("episode_return", np.float32),
    ("episode_length", np.int32), ("success", np.int32), ("timeout", np.int32),
    ("goals_reached", np.int32), ("dr_stand", np.float32), ("dr_joint_pose", np.float32),
    ("dr_torque", np.float32), ("dr_balance", np.float32), ("dr_progress", np.float32),
    ("nan", np.int32)])
assert EPISODE_STATS_DTYPE.itemsize == C.sizeof(SoloEpisodeStats)


def model_table(model: SoloModel) -> SoloModelTable:
    """Pack a :class:`SoloModel` into the C struct."""
    L = model.num_links
    if L > MAX_LINKS:
        raise ValueError(f"{L} links > SOLO_MAX_LINKS")
    t = SoloModelTable()
    t.abi_version = ABI_VERSION
    t.num_links = L
    for i in range(L):
        t.parent[i] = model.parent[i]
        t.jtype[i] = model.jtype[i]
        t.mass[i] = model.mass[i]
        for k in range(3):
            t.axis[i][k] = model.axis[i][k]
            t.origin[i][k] = model.origin[i][k]
            t.com[i][k] = model.com[i][k]
        for k in range(6):
            t.inertia[i][k] = model.inertia[i][k]
    t.base_mass = model.base_mass
    for k in range(3):
        t.base_com[k] = model.base_com[k]
    for k in range(6):
        t.base_inertia[k] = model.base_inertia[k]
    feet = model.feet_idx
    if len(feet) > MAX_FEET:
        raise ValueError("more than 4 feet")
    t.num_feet = len(feet)
    for f, l in enumerate(feet):
        t.foot_link[f] = l
        for k in range(3):
            t.foot_center[f][k] = model.foot_center[f][k]
    t.foot_radius = model.foot_radius
    return t


def default_params() -> SoloSimParams:
    """Reference defaults (solo.py:17-53, baseEnv.py:8-16, PyBullet defaults); must
    equal ``solo_default_params`` / ``oracle_default_params`` (tested)."""
    p = SoloSimParams()
    p.abi_version = ABI_VERSION
    p.dt = 1.0 / 240.0
    p.frame_skip = 4
    p.gravity_z = -9.81
    p.lin_damping = 0.04
    p.ang_damping = 0.04
    p.max_coord_vel = 100.0
    p.solver_iters = 50
    p.solver_residual_threshold = 1e-7
    p.contact_erp = 0.2
    p.contact_slop = 1e-5
    p.contact_margin = 0.02
    p.friction = 1.0
    p.cone_friction = 1
    p.torque_hold = 0
    p.control = CONTROL_TORQUE
    p.kp = 0.0
    p.kd = 0.0
    p.max_torque = 3.0
    p.joint_state_limit = 10.0
    p.joint_vel_limit = 100.0
    p.task = TASK_STAND
    p.episode_length = 400
    p.num_history_stack = 0
    p.initial_z = 0.35
    p.settle_min = 5
    p.settle_max = 12
    p.goal_radius = 2.0
    p.goal_reach_dist = 0.5
    p.pointgoal_dt = 4.0 / 240.0
    p.contact_flag_force = 0.2
    p.fall_z = 0.05
    p.stand_z = 0.2
    p.reset_mode = RESET_CACHED
    p.joint_limits = 1
    p.limit_rows_per_leg = 1
    p.joint_limit_erp = 0.2
    p.joint_limit_max_impulse = 100.0
    p.split_impulse_threshold = -0.04
    p.body_contacts = 0
    p.knee_radius = 0.015
    p.base_half_x, p.base_half_y = 0.2241, 0.1095
    p.base_z_lo, p.base_z_hi = -0.025, 0.028
    # randomised dynamics off; the ranges are only read with randomize = 1 (params_from_config sets them)
    p.randomize = 0
    p.friction_lo = p.friction_hi = 0.0
    p.base_mass_scale_lo = p.base_mass_scale_hi = 0.0
    p.motor_strength_lo = p.motor_strength_hi = 0.0
    # random pushes off (push_interval = 0); params_from_config sets all three
    p.push_force = 0.0
    p.push_interval = p.push_duration = 0
    return p


# config key -> (SoloSimParams range fields, nominal value (None: the params' friction), lower bound is exclusive)
_RANDOMIZE_KEYS = {
    "randomize_friction": ("friction_lo", "friction_hi", None, False),
    "randomize_base_mass": ("base_mass_scale_lo", "base_mass_scale_hi", 1.0, True),
    "randomize_motor_strength": ("motor_strength_lo", "motor_strength_hi", 1.0, True),
}


def _randomize_from_config(config: dict, p: SoloSimParams) -> None:
    """Per-env randomised dynamics: ``randomize_friction``, ``randomize_base_mass`` and
    ``randomize_motor_strength``, each ``[lo, hi]``.  Any of them present sets ``randomize``; a missing one
    keeps its value at the nominal (friction, 1, 1).  Malformed ranges raise ``ValueError``."""
    if not any(k in config for k in _RANDOMIZE_KEYS):
        return
    p.randomize = 1
    for key, (f_lo, f_hi, nominal, positive) in _RANDOMIZE_KEYS.items():
        if key not in config:
            v = p.friction if nominal is None else nominal
            setattr(p, f_lo, v)
            setattr(p, f_hi, v)
            continue
        r = config[key]
        try:
            lo, hi = (float(x) for x in r)
        except (TypeError, ValueError):
            raise ValueError(f"{key} must be a list [lo, hi] of two numbers, got {r!r}") from None
        if not (np.isfinite(lo) and np.isfinite(hi)) or lo > hi or lo < 0 or (positive and lo == 0):
            bound = "0 < lo <= hi" if positive else "0 <= lo <= hi"
            raise ValueError(f"{key}: [{lo}, {hi}] must satisfy {bound}")
        setattr(p, f_lo, lo)
        setattr(p, f_hi, hi)


_PUSH_KEYS = ("push_force", "push_interval", "push_duration")


def _push_from_config(config: dict, p: SoloSimParams) -> None:
    """Random pushes: ``push_force`` (N, >= 0), ``push_interval`` and ``push_duration`` (control steps,
    ``1 <= push_duration <= push_interval``).  ``push_force`` turns pushes on and needs the other two; a missing
    key or a malformed value raises ``ValueError``."""
    present = [k for k in _PUSH_KEYS if k in config]
    if not present:
        return
    if len(present) != len(_PUSH_KEYS):
        missing = [k for k in _PUSH_KEYS if k not in config]
        raise ValueError(f"random pushes need all of {', '.join(_PUSH_KEYS)}; missing {', '.join(missing)}")
    try:
        force = float(config["push_force"])
    except (TypeError, ValueError):
        raise ValueError(f"push_force must be a number, got {config['push_force']!r}") from None
    if not (np.isfinite(force) and force >= 0):
        raise ValueError(f"push_force must be finite and >= 0, got {force}")
    steps = {}
    for k in ("push_interval", "push_duration"):
        try:
            v = float(config[k])
        except (TypeError, ValueError):
            v = float("nan")
        if not (np.isfinite(v) and v == int(v)):
            raise ValueError(f"{k} must be a whole number of control steps, got {config[k]!r}")
        steps[k] = int(v)
    interval, duration = steps["push_interval"], steps["push_duration"]
    if interval < 1:
        raise ValueError(f"push_interval must be >= 1 when push_force is set, got {interval}")
    if not 1 <= duration <= interval:
        raise ValueError(f"push_duration must satisfy 1 <= push_duration <= push_interval ({interval}), "
                         f"got {duration}")
    if p.episode_length // interval >= 2 ** 30:
        raise ValueError("episode_length / push_interval must be below 2^30")
    p.push_force, p.push_interval, p.push_duration = force, interval, duration


def params_from_config(config: dict, model: Optional[SoloModel] = None) -> SoloSimParams:
    """Map a reference config dict onto ``SoloSimParams``.

    Keys and defaults are those of ``SoloBaseEnv.__init__`` (baseEnv.py:8-16):
    ``episode_length`` (required), ``frame_skip`` 4, ``control`` 'torque', ``task``
    'stand', ``gains`` None, ``num_history_stack`` 0, ``flat_ground`` True,
    ``use_treadmill`` False.  Extra keys (all default to the reference-faithful value):
    ``torque_hold``, ``solver_iters``, ``solver_residual_threshold``, ``contact_erp``, ``reset_mode``;
    ``randomize_friction``, ``randomize_base_mass``, ``randomize_motor_strength`` (per-env randomised
    dynamics, see ``_randomize_from_config``); ``push_force``, ``push_interval``, ``push_duration`` (random
    pushes on the base, see ``_push_from_config``).
    """
    p = default_params()
    p.episode_length = int(config["episode_length"])           # baseEnv.py:164 (required)
    p.frame_skip = int(config.get("frame_skip", 4))
    control = config.get("control", "torque")
    if control not in _CONTROL_NAMES:
        raise NotImplementedError(f"control {control!r}")       # solo.py:253-254
    p.control = _CONTROL_NAMES[control]
    task = config.get("task", "stand")
    if task not in _TASK_NAMES:
        raise NotImplementedError(f"task {task!r}")
    p.task = _TASK_NAMES[task]
    gains = config.get("gains", None)
    if p.control == CONTROL_PD:
        if gains is None:
            raise ValueError("control 'pd' needs gains: [Kp, Kd]")  # solo.py:240 unpacks None
        p.kp, p.kd = float(gains[0]), float(gains[1])
    p.num_history_stack = int(config.get("num_history_stack", 0))
    if not config.get("flat_ground", True):
        # simulation.py:130-136 raises for any non-flat ground in the reference (SURVEY §2)
        raise NotImplementedError("flat_ground: False is not supported (broken in the reference)")
    # use_treadmill: the treadmill strip is a static zero-dof body whose velocity is inert in
    # the contact solver (SURVEY §2); accepted and ignored.
    p.pointgoal_dt = p.frame_skip * p.dt
    if model is not None:
        p.joint_state_limit = model.joint_state_limit          # solo.py:109
    if model is not None and model.nj == 8:                    # base box extents per robot (SURVEY Appendix A)
        p.base_half_x, p.base_half_y = 0.212, 0.1046
    for k in ("torque_hold", "solver_iters", "cone_friction", "joint_limits", "limit_rows_per_leg", "settle_min",
              "settle_max", "body_contacts"):
        if k in config:
            setattr(p, k, int(config[k]))
    for k in ("contact_erp", "contact_margin", "contact_slop", "friction", "lin_damping",
              "ang_damping", "goal_radius", "solver_residual_threshold", "joint_limit_erp",
              "joint_limit_max_impulse", "split_impulse_threshold", "knee_radius", "base_half_x", "base_half_y",
              "base_z_lo", "base_z_hi"):
        if k in config:
            setattr(p, k, float(config[k]))
    rm = config.get("reset_mode", "cached")
    p.reset_mode = {"cached": RESET_CACHED, "simulate": RESET_SIMULATE}[rm]
    _randomize_from_config(config, p)
    _push_from_config(config, p)
    return p


def dims(model: SoloModel, p: SoloSimParams):
    """(nj, action dim, D0, D) — baseEnv.py:20-28, solo.py:186-222."""
    nj = model.nj
    act = nj + (2 if p.control == CONTROL_VPD else 0)
    d0 = 1 + 3 + 6 + 2 * nj + 4 + (4 if p.task == TASK_POINTGOAL else 0)
    return nj, act, d0, d0 * (1 + p.num_history_stack)
