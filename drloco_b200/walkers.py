"""Concrete walkers: which mocap rows feed which qpos/qvel entry, index sets, mirror tables.

Mirror of reference drloco/mujoco/mimic_walker3d.py, mimic_walker_165cm_65kg.py and drloco/mujoco/config.py.
"""
from __future__ import annotations

import dataclasses
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np

from . import config as cfgm
from .model import WalkerModel, get_model
from .ref_trajecs import straight_walk_trajecs as sw
from .ref_trajecs import loco3d_trajecs as l3
from .ref_trajecs.base_ref_trajecs import MocapTables, clip_weights as _clip_weights, concat_tables


def w3d_qpos_indices(n_rows: int = 38) -> List[int]:
    """reference mimic_walker3d.py:11-16."""
    tx, ty, tz = sw.trunk_euler_rows(n_rows)
    return [sw.COM_POSX, sw.COM_POSY, sw.COM_POSZ, tx, ty, tz,
            sw.HIP_SAG_ANG_R, sw.HIP_FRONT_ANG_R, sw.KNEE_ANG_R, sw.ANKLE_ANG_R,
            sw.HIP_SAG_ANG_L, sw.HIP_FRONT_ANG_L, sw.KNEE_ANG_L, sw.ANKLE_ANG_L]


def w3d_qvel_indices() -> List[int]:
    """reference mimic_walker3d.py:18-23."""
    return [sw.COM_VELX, sw.COM_VELY, sw.COM_VELZ, sw.TRUNK_ANGVEL_X, sw.TRUNK_ANGVEL_Y, sw.TRUNK_ANGVEL_Z,
            sw.HIP_SAG_ANGVEL_R, sw.HIP_FRONT_ANGVEL_R, sw.KNEE_ANGVEL_R, sw.ANKLE_ANGVEL_R,
            sw.HIP_SAG_ANGVEL_L, sw.HIP_FRONT_ANGVEL_L, sw.KNEE_ANGVEL_L, sw.ANKLE_ANGVEL_L]


# reference mimic_walker_165cm_65kg.py:6-15
W165_QPOS_INDICES = [l3.PELVIS_TX, l3.PELVIS_TZ, l3.PELVIS_TY, l3.PELVIS_LIST, l3.PELVIS_TILT, l3.PELVIS_ROTATION,
                     l3.LUMBAR_BENDING, l3.LUMBAR_EXTENSION, l3.LUMBAR_ROTATION,
                     l3.HIP_FLEXION_R, l3.HIP_ADDUCTION_R, l3.HIP_ROTATION_R, l3.KNEE_ANG_R, l3.ANKLE_ANG_R,
                     l3.HIP_FLEXION_L, l3.HIP_ADDUCTION_L, l3.HIP_ROTATION_L, l3.KNEE_ANG_L, l3.ANKLE_ANG_L]
W165_QVEL_INDICES = W165_QPOS_INDICES

# mirror tables (reference mimic_env.py:440-489)
MIRROR_OBS_IDX = [0, 1, 2, 3, 4, 5, 6, 11, 12, 13, 14, 7, 8, 9, 10, 15, 16, 17, 18, 19, 20, 25, 26, 27, 28, 21, 22, 23, 24]
MIRROR_OBS_NEG = [2, 4, 6, 8, 12, 16, 18, 20, 22, 26]
MIRROR_ACT_IDX = [4, 5, 6, 7, 0, 1, 2, 3]
MIRROR_ACT_NEG = [1, 5]


@dataclasses.dataclass
class WalkerSpec:
    cfg: cfgm.EnvConfig
    model: WalkerModel
    mocap: MocapTables
    com_indices: List[int]                 # _get_COM_indices
    trunk_rot_indices: List[int]           # _get_trunk_rot_joint_indices
    phase_joints: List[int]                # get_joint_indices_for_phase_estimation
    phase_from_cursor: bool                # mimic_env.py:416-419
    n_des_vel: int
    mirror: bool
    mocap_paths: Tuple[Optional[str], ...] = (None,)   # the file of every clip (None: the walker's default recording)

    @property
    def base_obs_dim(self) -> int:
        """the reference's observation (phase | desired velocity | qpos[1:] | qvel): DrlConfig.obs_dim, the width of
        the mirror tables"""
        return self.qpos_block + (self.model.nv - 1) + self.model.nv

    @property
    def qpos_block(self) -> int:
        """first column of the observation's qpos[1:] block"""
        return (1 if self.phase_from_cursor else 2 * len(self.phase_joints)) + self.n_des_vel

    @property
    def obs_dim(self) -> int:
        """the full row: the base observation, then one frame of nv - 1 reference qpos per EnvConfig.ref_obs_offsets"""
        return self.base_obs_dim + len(self.cfg.ref_obs_offsets) * (self.model.nv - 1)

    @property
    def act_dim(self) -> int:
        return self.model.nu

    @property
    def frame_skip(self) -> int:
        return self.cfg.frame_skip

    def mirror_tables(self):
        """(obs_idx, obs_sign, act_idx, act_sign) of the base observation; identity when mirroring is off."""
        D, A = self.base_obs_dim, self.act_dim
        oi, osn = np.arange(D, dtype=np.int32), np.ones(D, np.float32)
        ai, asn = np.arange(A, dtype=np.int32), np.ones(A, np.float32)
        if self.mirror:
            oi = np.array(MIRROR_OBS_IDX, np.int32)
            osn[MIRROR_OBS_NEG] = -1.0
            ai = np.array(MIRROR_ACT_IDX, np.int32)
            asn[MIRROR_ACT_NEG] = -1.0
        return oi, osn, ai, asn

    def ref_frame_mirror(self):
        """(idx, sign) [nv - 1] of a reference-pose frame: entry j of a mirrored frame is sign[j] * frame[idx[j]], the
        qpos-block part of the observation's mirror table (ref_frame_mirror_map)."""
        oi, osn, _, _ = self.mirror_tables()
        return ref_frame_mirror_map(oi, osn, self.qpos_block, self.model.nv - 1)


def ref_frame_mirror_map(obs_idx, obs_sign, block: int, n: int):
    """The part of an observation mirror table (obs[k] <- sign[k] * obs[idx[k]]) over the columns [block, block + n),
    relative to the block; ValueError when it reads a column outside the block (the map is not closed)."""
    idx = np.asarray(obs_idx, np.int64)[block:block + n] - block
    if idx.shape != (n,) or (idx < 0).any() or (idx >= n).any():
        raise ValueError(f"the mirror table does not map the qpos block [{block}, {block + n}) onto itself")
    return idx.astype(np.int32), np.asarray(obs_sign, np.float32)[block:block + n].copy()


def speed_profile(speeds, speed_profile_duration, control_freq) -> np.ndarray:
    """Desired walking speed per control step, as MimicEnv.activate_speed_control builds it (mimic_env.py:313-322):
    the profile is split into len(speeds)-1 regions of equal length, each a linspace between neighbouring speeds."""
    speeds = list(speeds)
    n_sections = len(speeds) - 1
    assert n_sections >= 1, "a speed profile needs at least two speeds"
    region = int(speed_profile_duration * control_freq / n_sections)
    return np.concatenate([np.linspace(speeds[i], speeds[i + 1], region) for i in range(n_sections)])


def _compile_mocap(cfg: cfgm.EnvConfig, mocap_path: Optional[str]) -> MocapTables:
    """One recording -> its tables (reference drloco/mujoco/config.py:9-10 ``env_map`` and the walkers' refs)."""
    if cfg.env_id == cfgm.STRAIGHT_WALKER:
        rows, _ = sw.load_steps(mocap_path or sw.PATH_CONSTANT_SPEED)
        return sw.StraightWalkingTrajectories(w3d_qpos_indices(rows.shape[0]), w3d_qvel_indices(),
                                              path=mocap_path).tables()
    if cfg.env_id == cfgm.WALKER_165:
        return l3.Loco3dReferenceTrajectories(W165_QPOS_INDICES, W165_QVEL_INDICES, {}, path=mocap_path,
                                              control_freq=cfg.ctrl_freq).tables()
    raise KeyError(cfg.env_id)


def make_spec(cfg: Optional[cfgm.EnvConfig] = None, mocap_path: Union[None, str, Sequence[Optional[str]]] = None,
              clip_weights=None) -> WalkerSpec:
    """env id -> everything the device needs (reference drloco/mujoco/config.py:9-10 ``env_map``).

    ``mocap_path``: one recording (None: the walker's default), or a sequence of them, a mocap library whose clips an
    episode never leaves (concat_tables).  ``clip_weights``: one RSI weight per clip (finite, >= 0, positive sum);
    None weighs the clips by their sample counts.  A library of one path is the single recording, bit for bit."""
    cfg = cfg or cfgm.EnvConfig()
    model = get_model(cfg.env_id)
    paths = (mocap_path,) if mocap_path is None or isinstance(mocap_path, str) else tuple(mocap_path)
    if not paths:
        raise ValueError("make_spec: mocap_path is an empty sequence")
    if cfg.env_id not in (cfgm.STRAIGHT_WALKER, cfgm.WALKER_165):
        raise KeyError(cfg.env_id)
    clips = [_compile_mocap(cfg, p) for p in paths]
    if len(clips) == 1:
        _clip_weights(clip_weights, [clips[0].n_samples])     # validated; one clip is always drawn
        mocap = clips[0]
    else:
        mocap = concat_tables(clips, clip_weights)
    if cfg.env_id == cfgm.STRAIGHT_WALKER:
        return WalkerSpec(cfg, model, mocap, [0, 1, 2], [3, 4, 5], [6, 8, 10, 12], True, 1,
                          cfg.is_mod(cfgm.MOD_MIRR_POLICY), paths)
    return WalkerSpec(cfg, model, mocap, [0, 1, 2], [3, 4, 5], [9, 12, 14, 17], False, 2, False, paths)
