"""Base class of the reference-trajectory *table compilers*.

In the reference, ``BaseReferenceTrajectories`` (drloco/ref_trajecs/base_ref_trajecs.py:6-158) is a per-env CPU
cursor over a (rows x samples) matrix: ``next()`` advances ``_pos``, ``get_qpos()/get_qvel()`` gather the rows the
walker needs.  On the B200 the cursor lives in device memory, one per environment, and is advanced inside the fused
step kernel; the classes here keep the reference's names and constructor signatures but only *compile* the mocap
into the flat tables the kernels index:

    ref  float [n_samples, 2*nv]   qpos rows then qvel rows, already gathered in model order (base:44-56)
    step_off / step_len            where each mocap step starts and how long it is (1 step for loco3d)

The per-env cursor logic itself is restated once for tests in ``oracle/env_oracle.py`` and once for the GPU in
``csrc/mimic_step.cu``.
"""
from __future__ import annotations

import dataclasses
import os
from typing import Dict, Optional, Sequence

import numpy as np

DATA_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "data")

# cursor advance rules (SURVEY.md Q6)
CURSOR_STEPWISE = 0   # StraightWalkingTrajectories.next (straight_walk_trajecs.py:141-159)
CURSOR_WRAP = 1       # BaseReferenceTrajectories.next (base_ref_trajecs.py:95-103)


@dataclasses.dataclass
class MocapTables:
    """Everything the device (and the oracle) needs to know about one mocap."""
    cursor_mode: int
    increment: int                 # samples per control step (base:87-93)
    ref: np.ndarray                # float64 [n_samples, 2*nv]
    step_off: np.ndarray           # int32 [n_steps]
    step_len: np.ndarray           # int32 [n_steps]
    left_step: np.ndarray          # uint8 [n_steps]  (straight:221-230)
    step_vel: np.ndarray           # float64 [n_steps] smoothed mean COM-X velocity per step (straight:393-415)
    step_last_comx: np.ndarray     # float64 [n_steps] COM-X at the last sample of each step (straight:339)
    com_z_col: int                 # column of ``ref`` holding the COM-Z position (straight:482, loco3d:48)
    des_vel_prefix: Optional[np.ndarray] = None   # float64 [n_samples+1, 2] prefix sums for loco3d:51-68
    des_vel_window: int = 0
    des_vel_rows: Optional[np.ndarray] = None     # float64 [2, n_samples] the velocity rows themselves (the oracle
                                                  # takes np.mean of the slice exactly like loco3d:62-68)
    # mocap library (concat_tables): clip k = steps [clip_first_step[k], clip_first_step[k + 1]), drawn at RSI with
    # probability clip_weight[k]; a single recording is one clip of weight 1
    clip_first_step: Optional[np.ndarray] = None  # int32 [n_clips + 1]
    clip_weight: Optional[np.ndarray] = None      # float64 [n_clips], sums to 1

    def __post_init__(self):
        if self.clip_first_step is None:
            self.clip_first_step = np.array([0, self.n_steps], np.int32)
        if self.clip_weight is None:
            self.clip_weight = np.ones(1)

    @property
    def n_steps(self) -> int:
        return int(self.step_len.shape[0])

    @property
    def n_samples(self) -> int:
        return int(self.ref.shape[0])

    @property
    def n_clips(self) -> int:
        return int(self.clip_first_step.shape[0]) - 1


def clip_weights(weights, n_samples) -> np.ndarray:
    """Normalised RSI clip weights: ``weights`` (finite, >= 0, positive sum, one per clip), or None for weights
    proportional to the clips' sample counts ``n_samples``."""
    n_samples = np.asarray(n_samples, np.float64)
    w = n_samples if weights is None else np.asarray(weights, np.float64).reshape(-1)
    if w.shape != n_samples.shape:
        raise ValueError(f"clip_weights: need one weight per clip ({n_samples.size}), got {w.size}")
    if not np.all(np.isfinite(w)) or np.any(w < 0) or not w.sum() > 0:
        raise ValueError(f"clip_weights must be finite and >= 0 with a positive sum, got {w.tolist()}")
    return w / np.add.accumulate(w)[-1]          # summed in order, as drl_set_mocap_clips does


def concat_tables(clips: Sequence[MocapTables], weights=None) -> MocapTables:
    """A mocap library: the single-recording tables ``clips`` one after the other.  Step offsets are shifted by the
    samples before each clip; the per-step tables and, in wrap mode, the desired-velocity prefix sums (which restart at
    every clip) and rows are concatenated.  ``weights``: see clip_weights.  Every clip keeps the row map it was compiled
    with (a 38-row and a 40-row straight-walking file can share a library).  Raises for an empty list, a clip that is
    itself a library, mixed cursor modes, increments, COM-Z columns, desired-velocity windows or widths, a
    stepwise clip of fewer than 2 steps or a wrap-mode clip of other than 1 step."""
    clips = list(clips)
    if not clips:
        raise ValueError("concat_tables: no clips")
    t0 = clips[0]
    for k, t in enumerate(clips):
        if t.n_clips != 1:
            raise ValueError(f"concat_tables: clip {k} is already a library of {t.n_clips} clips")
        for name in ("cursor_mode", "increment", "com_z_col", "des_vel_window"):
            if getattr(t, name) != getattr(t0, name):
                raise ValueError(f"concat_tables: clip {k} has {name} {getattr(t, name)}, clip 0 has {getattr(t0, name)}")
        if t.ref.shape[1] != t0.ref.shape[1]:
            raise ValueError(f"concat_tables: clip {k} has {t.ref.shape[1]} reference columns, clip 0 {t0.ref.shape[1]}")
        if t.cursor_mode == CURSOR_STEPWISE and t.n_steps < 2:
            raise ValueError(f"concat_tables: clip {k} has {t.n_steps} steps; the per-clip wrap "
                             "(straight_walk_trajecs.py:330-333) needs at least 2")
        if t.cursor_mode == CURSOR_WRAP and t.n_steps != 1:
            raise ValueError(f"concat_tables: wrap-mode clip {k} has {t.n_steps} steps, not 1")
    n_samples = np.array([t.n_samples for t in clips], np.int64)
    sample0 = np.concatenate([[0], np.cumsum(n_samples)[:-1]])
    wrap = t0.cursor_mode == CURSOR_WRAP
    return MocapTables(
        cursor_mode=t0.cursor_mode, increment=t0.increment, ref=np.concatenate([t.ref for t in clips]),
        step_off=np.concatenate([t.step_off + s0 for t, s0 in zip(clips, sample0)]).astype(np.int32),
        step_len=np.concatenate([t.step_len for t in clips]).astype(np.int32),
        left_step=np.concatenate([t.left_step for t in clips]).astype(np.uint8),
        step_vel=np.concatenate([t.step_vel for t in clips]),
        step_last_comx=np.concatenate([t.step_last_comx for t in clips]), com_z_col=t0.com_z_col,
        des_vel_prefix=np.concatenate([t.des_vel_prefix for t in clips]) if wrap else None,
        des_vel_window=t0.des_vel_window,
        des_vel_rows=np.concatenate([t.des_vel_rows for t in clips], axis=1) if wrap else None,
        clip_first_step=np.concatenate([[0], np.cumsum([t.n_steps for t in clips])]).astype(np.int32),
        clip_weight=clip_weights(weights, n_samples))


class BaseReferenceTrajectories:
    """Same constructor as the reference (base_ref_trajecs.py:20-42); subclasses provide ``_load_ref_trajecs``."""

    def __init__(self, sample_freq, control_freq, qpos_indices, qvel_indices, data_labels=(), adaptations=None):
        self._sample_freq = sample_freq
        self._control_freq = control_freq
        self._qpos_indices = list(qpos_indices)
        self._qvel_indices = list(qvel_indices)
        self._qlabels = data_labels
        self._qpos_full, self._qvel_full = self._load_ref_trajecs()
        self._n_joints, self._trajec_len = self._qpos_full.shape
        self.adapt_trajectories(adaptations or {})
        if not (len(data_labels) == 0 or len(data_labels) in (self._n_joints, len(self._qpos_indices))):
            raise AssertionError(
                "Please provide a label for each row in the data matrix.\n"
                f"You provided {len(data_labels)} labels for a matrix of shape {self._qpos_full.shape}.\n")
        self._set_increment()

    def _set_increment(self):
        increment = self._sample_freq / self._control_freq
        if not float(increment).is_integer():
            raise AssertionError(
                "Please check your control frequency and the sample frequency of the reference data!"
                f"The sampling frequency ({self._sample_freq}) of the reference data should be equal to "
                f"or an integer multiple of the control frequency which is set to {self._control_freq}.")
        self._increment = int(increment)

    def adapt_trajectories(self, adaptations_dict: Dict[int, float]):
        """Scale individual rows (base_ref_trajecs.py:105-118)."""
        for index, scalar in adaptations_dict.items():
            self._qpos_full[index, :] *= scalar
            if self._qvel_full is not self._qpos_full:
                self._qvel_full[index, :] *= scalar

    def get_kinematics_labels(self):
        return self._qlabels

    # ---- to override -------------------------------------------------------------------------
    def _load_ref_trajecs(self):
        raise NotImplementedError

    def _get_COM_Z_pos_index(self) -> int:
        raise NotImplementedError

    def tables(self) -> MocapTables:
        raise NotImplementedError


def gather(rows: np.ndarray, idx: Sequence[int]) -> np.ndarray:
    """rows [R, T] -> [T, len(idx)] (the reference's fancy index ``full[indices, pos]`` for every pos)."""
    return np.ascontiguousarray(rows[list(idx), :].T)
