"""Configuration of the batched DeepMimic environment.

Mirror of the step-path fields of reference drloco/config/config.py and drloco/config/hypers.py.  The reference keeps
them as import-time module constants; here they are one dataclass so that several configurations can coexist in a
process (tests, benchmarks), with the reference's values as defaults.
"""
from __future__ import annotations

import dataclasses
from typing import Tuple

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
