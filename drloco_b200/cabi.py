"""ctypes mirror of include/drloco_b200.h (struct layouts and enum values) — the reference-side binding.

A DRLoco maintainer binds libdrloco_b200.so exactly like this (see INTEGRATION.md); no torch types cross the boundary,
only raw pointers and sizes.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

DRL_ABI_VERSION = 4
MAX_DOF, MAX_BODY, MAX_ACT, MAX_SPHERE, MAX_BOX, MAX_SITE, MAX_OBS, MAX_PHASE_JOINTS = 24, 12, 16, 16, 8, 16, 64, 4
MAX_EE = 4
MAX_REF_OBS = 3        # DRL_MAX_REF_OBS: reference-pose frames of drl_set_ref_obs (EnvConfig.ref_obs_offsets)
INTEGRATOR_RK4, INTEGRATOR_EULER = 0, 1
CURSOR_STEPWISE, CURSOR_WRAP = 0, 1
PHASE_FROM_CURSOR, PHASE_FROM_JOINTS = 0, 1
ACTUATION_TORQUE, ACTUATION_PD = 0, 1
EXTRA_NAMES = ("pos_rew", "vel_rew", "com_rew", "walked_distance", "mean_abs_torque", "des_vel", "phase", "z_offset",
               "ep_len_smoothed", "ep_ret_smoothed", "mean_reward_smoothed", "mean_ep_pos_rew_smoothed",
               "mean_ep_vel_rew_smoothed", "mean_ep_com_rew_smoothed", "moved_distance", "mean_abs_ep_torque_smoothed")
EXTRA_COUNT = 16
STAT_NAMES = ("episodes", "ep_len_sum", "ep_ret_sum", "ep_mean_rew_sum", "pos_rew_sum", "vel_rew_sum", "com_rew_sum",
              "rew_steps", "moved_distance_sum", "abs_torque_sum", "env_steps", "blowups", "falls", "timeouts",
              "solver_iters", "dyn_evals", "solver_capped", "et_com_low", "et_trunk", "et_drunk")
STATS_COUNT = 20

d, i32 = C.c_double, C.c_int32


class DrlWalkerModel(C.Structure):
    _fields_ = [
        ("nv", i32), ("nb", i32), ("nu", i32), ("n_sphere", i32), ("n_box", i32), ("n_site", i32),
        ("timestep", d), ("gravity_z", d), ("solref", d * 2), ("solimp", d * 5),
        ("body_parent", i32 * MAX_BODY), ("body_pos", d * 3 * MAX_BODY), ("body_mass", d * MAX_BODY),
        ("body_ipos", d * 3 * MAX_BODY), ("body_inertia", d * 3 * MAX_BODY), ("body_invweight0", d * 2 * MAX_BODY),
        ("dof_body", i32 * MAX_DOF), ("dof_type", i32 * MAX_DOF), ("dof_axis_idx", i32 * MAX_DOF),
        ("dof_axis_sign", d * MAX_DOF), ("dof_ref", d * MAX_DOF), ("dof_damping", d * MAX_DOF),
        ("dof_armature", d * MAX_DOF), ("dof_limited", i32 * MAX_DOF), ("dof_range", d * 2 * MAX_DOF),
        ("dof_invweight0", d * MAX_DOF),
        ("act_dof", i32 * MAX_ACT), ("act_gear", d * MAX_ACT), ("act_ctrlrange", d * 2 * MAX_ACT),
        ("act_forcerange", d * 2 * MAX_ACT),
        ("sphere_body", i32 * MAX_SPHERE), ("sphere_pos", d * 3 * MAX_SPHERE), ("sphere_radius", d * MAX_SPHERE),
        ("sphere_mu", d * MAX_SPHERE),
        ("box_body", i32 * MAX_BOX), ("box_center", d * 3 * MAX_BOX), ("box_corner", d * 3 * 8 * MAX_BOX),
        ("box_mu", d * MAX_BOX),
        ("site_body", i32 * MAX_SITE), ("site_pos", d * 3 * MAX_SITE),
        ("n_ee", i32), ("ee_body", i32 * MAX_EE), ("ee_pos", d * 3 * MAX_EE),
    ]


class DrlConfig(C.Structure):
    _fields_ = [
        ("num_envs", i32), ("device", i32), ("frame_skip", i32), ("integrator", i32), ("ep_dur_max", i32),
        ("mirror_policy", i32), ("phase_mode", i32), ("n_phase_joints", i32), ("phase_joints", i32 * MAX_PHASE_JOINTS),
        ("eval_n_times", i32),
        ("ctrl_freq", d), ("rew_weights", d * 4), ("rew_scale", d), ("alive_bonus", d), ("fall_z", d),
        ("seed", C.c_uint64), ("env_id_offset", C.c_int64),
        ("obs_dim", i32), ("act_dim", i32),
        ("mirror_obs_idx", i32 * MAX_OBS), ("mirror_obs_sign", C.c_float * MAX_OBS),
        ("mirror_act_idx", i32 * MAX_ACT), ("mirror_act_sign", C.c_float * MAX_ACT),
        ("lanes_per_env", i32), ("early_termination", i32), ("monitor_median_torque", i32),
        ("ee_weight", d), ("ee_scale", d),
    ]


def _fill(dst, src):
    """copy a numpy array into a (possibly nested) ctypes array, zero padded."""
    a = np.ctypeslib.as_array(dst)
    a[...] = 0
    src = np.asarray(src)
    if src.size:
        a[tuple(slice(0, n) for n in src.shape)] = src


def pack_model(m) -> DrlWalkerModel:
    """drloco_b200.model.WalkerModel -> DrlWalkerModel."""
    from .model import GRAVITY_Z, SOLREF, SOLIMP
    if m.nv > MAX_DOF or m.nb > MAX_BODY or m.nu > MAX_ACT or len(m.sphere_body) > MAX_SPHERE \
            or len(m.box_body) > MAX_BOX or len(m.site_body) > MAX_SITE or len(m.ee_body) > MAX_EE:
        raise ValueError("model exceeds the fixed capacities of DrlWalkerModel")
    s = DrlWalkerModel()
    s.nv, s.nb, s.nu = m.nv, m.nb, m.nu
    s.n_sphere, s.n_box, s.n_site = len(m.sphere_body), len(m.box_body), len(m.site_body)
    s.n_ee = len(m.ee_body)
    s.timestep, s.gravity_z = m.timestep, GRAVITY_Z
    _fill(s.solref, SOLREF)
    _fill(s.solimp, SOLIMP)
    for name in ("body_parent", "body_pos", "body_mass", "body_ipos", "body_inertia", "body_invweight0", "dof_body",
                 "dof_type", "dof_axis_idx", "dof_axis_sign", "dof_ref", "dof_damping", "dof_armature", "dof_limited",
                 "dof_range", "dof_invweight0", "act_dof", "act_gear", "act_ctrlrange", "act_forcerange", "sphere_body",
                 "sphere_pos", "sphere_radius", "sphere_mu", "box_body", "box_center", "box_corner", "box_mu",
                 "site_body", "site_pos", "ee_body", "ee_pos"):
        _fill(getattr(s, name), getattr(m, name))
    return s
