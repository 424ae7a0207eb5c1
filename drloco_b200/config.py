"""Configuration of the batched DeepMimic environment.

Mirror of the step-path fields of reference drloco/config/config.py and drloco/config/hypers.py.  The reference keeps
them as import-time module constants; here they are one dataclass so that several configurations can coexist in a
process (tests, benchmarks), with the reference's values as defaults.
"""
from __future__ import annotations

import dataclasses
import math
from typing import Optional, Tuple, Union

import numpy as np

from .cabi import MAX_REF_OBS   # reference-pose frames (DRL_MAX_REF_OBS)

# environment ids (reference drloco/mujoco/config.py:5-6)
STRAIGHT_WALKER = "StraightMimicWalker"
WALKER_165 = "MimicWalker165cm65kg"

# control / simulation frequency per env (reference config.py:20-21, mujoco/config.py:13-14)
CTRL_FREQS = {STRAIGHT_WALKER: 200, WALKER_165: 100}
SIM_FREQS = {STRAIGHT_WALKER: 1000, WALKER_165: 1000}

# modification flags (reference hypers.py:13-29)
MOD_CUSTOM_POLICY = "cstm_pi"
MOD_CLIPRANGE_SCHED = "clip_sched"
MOD_MIRR_POLICY = "mirr_py"


@dataclasses.dataclass
class EnvConfig:
    env_id: str = STRAIGHT_WALKER                       # config.py:18
    ctrl_freq: int = 0                                  # 0 -> CTRL_FREQS[env_id]
    eval_n_times: int = 20                              # config.py:23
    min_stable_distance: float = 15.0                   # config.py:25
    modifications: Tuple[str, ...] = (MOD_CUSTOM_POLICY, MOD_MIRR_POLICY)   # hypers.py:23
    rew_weights: Tuple[float, float, float, float] = (0.8, 0.2, 0.0, 0.0)  # hypers.py:48 (pos, vel, com, energy)
    rew_scale: float = 1.0                              # hypers.py:51
    alive_bonus: float = 0.2                            # hypers.py:55 (0.2 * rew_scale)
    ep_dur_max: int = 3000                              # hypers.py:58
    fall_z: float = 0.5                                 # mimic_env.py:120
    early_termination: bool = False                     # True: do_terminate_early (mimic_env.py:652-702) also ends the
                                                        # episode; the reference never does (mimic_env.py:120-123)
    median_torque: bool = False                         # True: keep the per-episode torque history behind Monitor's
                                                        # median_abs_torque_smoothed (monitor_wrapper.py:131; 4 *
                                                        # ep_dur_max bytes per env and a radix-select median at every
                                                        # episode end).  The reference's callback never reads it.
    ee_weight: float = 0.0                              # DeepMimic end-effector (foot position) reward term, added to
                                                        # the imitation reward with this weight; 0 = off, as in the
                                                        # reference (see README "End-effector reward")
    ee_scale: float = 40.0                              # ee_rew = exp(-ee_scale * sum of squared foot-position errors)
    actuation: str = "torque"                           # "torque": the action is the motor force (the reference);
                                                        # "pd": every motor is a position servo, MuJoCo <position kp kv>,
                                                        # and the action picks its target in the joint's range (see
                                                        # README "PD actuation")
    pd_kp: Union[None, float, Tuple[float, ...]] = None   # servo stiffness, > 0: one value for every actuator or one
                                                        # per actuator in actuator order; required with "pd"
    pd_kv: Union[None, float, Tuple[float, ...]] = None   # servo damping, >= 0, as pd_kp; None = 0 (MuJoCo's default)
    contact_termination: bool = False                   # DeepMimic early termination: the episode also ends when a
                                                        # body other than the feet touches the floor; off = the
                                                        # reference (see README "Contact termination")
    adaptive_rsi: float = 0.0                           # failure-weighted RSI: the share (0 < lambda <= 1) of random
                                                        # RSI draws that favour the mocap phases where episodes end
                                                        # early; 0 = off, the reference's uniform draw (see README
                                                        # "Failure-weighted RSI")
    adaptive_rsi_halflife: int = 2000                   # half-life of its per-phase counts, in control steps of the
                                                        # batch (a choice, not a tuned value)
    ref_obs_offsets: Tuple[int, ...] = ()               # reference-pose observations: one frame of reference qpos[1:]
                                                        # per offset (control steps ahead, ints in [1, 256], strictly
                                                        # increasing, at most 3) appended to the observation; () = off,
                                                        # the reference's layout (see README "Reference-pose
                                                        # observations")
    gamma: float = 0.0                                  # 0 -> by ctrl_freq, hypers.py:68
    integrator: str = "rk4"                             # xml:11; "euler" = MuJoCo semi-implicit Euler (fast mode)
    seed: int = 33                                      # utils.py:97

    def __post_init__(self):
        if self.ctrl_freq == 0:
            self.ctrl_freq = CTRL_FREQS[self.env_id]
        if self.gamma == 0.0:
            self.gamma = {50: 0.99, 100: 0.99, 200: 0.995, 400: 0.998}[self.ctrl_freq]
        if self.env_id == WALKER_165 and self.is_mod(MOD_MIRR_POLICY):
            # mirroring is only defined for the straight walker (hypers.py:31-39; loco3d refs have no is_step_left)
            self.modifications = tuple(m for m in self.modifications if m != MOD_MIRR_POLICY)
        if self.actuation not in ("torque", "pd"):
            raise ValueError(f"actuation must be 'torque' or 'pd', got {self.actuation!r}")
        if self.actuation == "torque":
            if self.pd_kp is not None or self.pd_kv is not None:
                raise ValueError("pd_kp / pd_kv are the gains of actuation='pd'; the torque mode has none")
        else:
            if self.pd_kp is None:
                raise ValueError("actuation='pd' needs pd_kp (there are no default gains)")
            self.pd_gains()
        lam = self.adaptive_rsi
        if isinstance(lam, bool) or not isinstance(lam, (int, float, np.integer, np.floating)) or not (0.0 <= lam <= 1.0):
            raise ValueError(f"adaptive_rsi must be a number in [0, 1], got {lam!r}")
        hl = self.adaptive_rsi_halflife
        if isinstance(hl, bool) or not isinstance(hl, (int, np.integer)) or hl <= 0 or hl >= 2 ** 31:
            raise ValueError(f"adaptive_rsi_halflife must be a positive int32 number of control steps, got {hl!r}")
        offs = self.ref_obs_offsets
        if isinstance(offs, (str, bytes)) or not isinstance(offs, (tuple, list)):
            raise ValueError(f"ref_obs_offsets must be a tuple of ints, got {offs!r}")
        if len(offs) > MAX_REF_OBS:
            raise ValueError(f"ref_obs_offsets: at most {MAX_REF_OBS} frames, got {len(offs)}")
        for k in offs:
            if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or not 1 <= k <= 256:
                raise ValueError(f"ref_obs_offsets: every offset must be an int in [1, 256], got {offs!r}")
        if any(b <= a for a, b in zip(offs, offs[1:])):
            raise ValueError(f"ref_obs_offsets must be strictly increasing, got {offs!r}")
        self.ref_obs_offsets = tuple(int(k) for k in offs)

    def pd_gains(self, nu: Optional[int] = None) -> Tuple[np.ndarray, np.ndarray]:
        """(kp, kv) of actuation='pd' as float64 arrays in actuator order, scalars broadcast to the walker's nu
        actuators; raises ValueError for a wrong length or a gain out of range (kp finite and > 0, kv finite and >= 0)."""
        if nu is None:
            from .model import get_model
            nu = get_model(self.env_id).nu

        def per_actuator(x, name):
            a = np.full(nu, float(x)) if np.ndim(x) == 0 else np.array([float(g) for g in x], np.float64)
            if a.shape != (nu,):
                raise ValueError(f"{name}: {a.size} gains for {nu} actuators")
            return a
        kp = per_actuator(self.pd_kp, "pd_kp")
        kv = per_actuator(0.0 if self.pd_kv is None else self.pd_kv, "pd_kv")
        if not all(math.isfinite(g) and g > 0.0 for g in kp):
            raise ValueError(f"pd_kp must be finite and > 0, got {self.pd_kp}")
        if not all(math.isfinite(g) and g >= 0.0 for g in kv):
            raise ValueError(f"pd_kv must be finite and >= 0, got {self.pd_kv}")
        return kp, kv

    def is_mod(self, mod_str: str) -> bool:
        """reference hypers.py:26-29 (substring test on the joined modification string)."""
        return mod_str in "/".join(self.modifications)

    @property
    def frame_skip(self) -> int:
        """reference mimic_env.py:194-207."""
        skip = SIM_FREQS[self.env_id] / self.ctrl_freq
        if not float(skip).is_integer():
            raise AssertionError("The simulation frequency should be an integer multiple of the control frequency.")
        return int(skip)
