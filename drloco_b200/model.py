"""Walker model compiler: MJCF subset -> flat POD tables for the oracle and the CUDA kernels.

The reference defines its walkers as MuJoCo MJCF files and lets MuJoCo compile them
(reference: drloco/mujoco/xml/walker3d_flat_feet.xml, drloco/mujoco/xml/walker_165cm_65kg.xml,
loaded at drloco/mujoco/mimic_env.py:52 through gym's MujocoEnv).  This module restates the part of
MuJoCo's model compiler those two files exercise:

* kinematic tree of bodies with explicit inertials (``inertiafromgeom="false"``),
* 1-DoF slide / hinge joints whose axes are +-coordinate axes and whose anchor is the body origin,
* motors with ctrl/force ranges, plane-vs-{box, capsule} collision geometry, foot-corner sites,
* the compile-time constants MuJoCo derives at ``qpos0``: ``dof_invweight0`` and ``body_invweight0``
  (used by the soft-constraint regulariser, SURVEY.md Appendix A).

Two sources feed the same ``WalkerModel``: the built-in specs below (numbers transcribed from the
XML lines cited next to them) and ``load_mjcf(path)`` for a user-supplied file.  ``tests/`` checks they agree
whenever the reference checkout is present.
"""
from __future__ import annotations

import dataclasses
import math
import xml.etree.ElementTree as ET
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

SLIDE, HINGE = 0, 1

# MuJoCo defaults that the reference XMLs leave untouched (SURVEY.md Appendix A).
GRAVITY_Z = -9.81
SOLREF = (0.02, 1.0)                     # timeconst, dampratio
SOLIMP = (0.9, 0.95, 0.001, 0.5, 2.0)    # d0, dmax, width, midpoint, power
FLOOR_FRICTION = 0.7                     # floor inherits the default class friction ".7 .1 .1"
MJ_MINVAL = 1e-15


@dataclasses.dataclass
class WalkerModel:
    """Flat description of one walker.  Bodies exclude the world body; ``parent == -1`` is the world."""
    name: str
    timestep: float
    # bodies
    body_names: List[str]
    body_parent: np.ndarray      # [nb] int32
    body_pos: np.ndarray         # [nb,3] offset of the body frame in the parent frame
    body_mass: np.ndarray        # [nb]
    body_ipos: np.ndarray        # [nb,3] centre of mass in the body frame
    body_inertia: np.ndarray     # [nb,3] diagonal inertia about the COM, body axes
    # dofs (== joints, all 1-DoF, nq == nv)
    dof_names: List[str]
    dof_body: np.ndarray         # [nv] int32
    dof_type: np.ndarray         # [nv] int32  SLIDE / HINGE
    dof_axis_idx: np.ndarray     # [nv] int32  0/1/2 coordinate axis of the body frame
    dof_axis_sign: np.ndarray    # [nv] +1/-1
    dof_ref: np.ndarray          # [nv] qpos0
    dof_damping: np.ndarray      # [nv]
    dof_armature: np.ndarray     # [nv]
    dof_limited: np.ndarray      # [nv] uint8
    dof_range: np.ndarray        # [nv,2]
    # actuators (motors)
    act_names: List[str]
    act_dof: np.ndarray          # [nu] int32
    act_gear: np.ndarray         # [nu]
    act_ctrlrange: np.ndarray    # [nu,2]
    act_forcerange: np.ndarray   # [nu,2]
    # collision geometry against the floor plane z = 0
    sphere_body: np.ndarray      # [ns] int32 (capsule end spheres)
    sphere_pos: np.ndarray       # [ns,3] body frame
    sphere_radius: np.ndarray    # [ns]
    sphere_mu: np.ndarray        # [ns] contact friction = max(floor, geom)
    box_body: np.ndarray         # [nx] int32
    box_center: np.ndarray       # [nx,3] body frame
    box_corner: np.ndarray       # [nx,8,3] corner relative to the box centre, body frame, MuJoCo corner order
    box_mu: np.ndarray           # [nx]
    # foot-corner sites used by reset (reference: mimic_env.py:546-559)
    site_body: np.ndarray        # [nsite] int32
    site_pos: np.ndarray         # [nsite,3]
    # end-effector points of the optional DeepMimic end-effector reward: the centre of every box geom on a leaf body
    # that does not hang directly from the root (a leaf on the root, like walker_165cm_65kg's torso, is a trunk
    # segment, not the end of a limb).  Both walkers: the two foot boxes.
    ee_body: np.ndarray = None           # [n_ee] int32
    ee_pos: np.ndarray = None            # [n_ee,3] body frame
    # compile-time constants at qpos0
    dof_invweight0: np.ndarray = None    # [nv]
    body_invweight0: np.ndarray = None   # [nb,2] translational, rotational

    @property
    def nv(self) -> int:
        return int(self.dof_body.shape[0])

    @property
    def nb(self) -> int:
        return int(self.body_parent.shape[0])

    @property
    def nu(self) -> int:
        return int(self.act_dof.shape[0])

    @property
    def qpos0(self) -> np.ndarray:
        return self.dof_ref.copy()

    @property
    def total_mass(self) -> float:
        return float(self.body_mass.sum())


# ----------------------------------------------------------------------------------------------
# float64 reference kinematics / mass matrix used ONLY for the compile-time constants
# (MuJoCo computes these once in mj_setConst; they are model data, not part of the step path).
# ----------------------------------------------------------------------------------------------

def _rot_axis(k: int, ang: float) -> np.ndarray:
    c, s = math.cos(ang), math.sin(ang)
    R = np.eye(3)
    i, j = (k + 1) % 3, (k + 2) % 3
    R[i, i], R[i, j], R[j, i], R[j, j] = c, -s, s, c
    return R


def forward_kinematics(m: WalkerModel, q: np.ndarray):
    """MuJoCo mj_kinematics restricted to this model class.

    Joints of one body are applied in declaration order; a hinge rotates about its axis expressed in the
    body frame *as already rotated by the earlier joints of that body*; slides translate along the axis in
    the same way.  Returns (xpos[nb,3], xmat[nb,3,3], axis_w[nv,3], anchor[nv,3]).
    """
    nb, nv = m.nb, m.nv
    xpos = np.zeros((nb, 3))
    xmat = np.zeros((nb, 3, 3))
    axis_w = np.zeros((nv, 3))
    anchor = np.zeros((nv, 3))
    dofs_of = [[j for j in range(nv) if m.dof_body[j] == b] for b in range(nb)]
    for b in range(nb):
        p = int(m.body_parent[b])
        if p < 0:
            pos, R = m.body_pos[b].copy(), np.eye(3)
        else:
            pos, R = xpos[p] + xmat[p] @ m.body_pos[b], xmat[p].copy()
        for j in dofs_of[b]:
            k, sg = int(m.dof_axis_idx[j]), float(m.dof_axis_sign[j])
            axis_w[j] = sg * R[:, k]
            anchor[j] = pos
            d = q[j] - m.dof_ref[j]
            if m.dof_type[j] == SLIDE:
                pos = pos + axis_w[j] * d
            else:
                R = R @ _rot_axis(k, sg * d)
        xpos[b], xmat[b] = pos, R
    return xpos, xmat, axis_w, anchor


def body_jacobians(m: WalkerModel, q: np.ndarray, point_local: Optional[np.ndarray] = None):
    """(jacp[nb,3,nv], jacr[nb,3,nv]) of the point ``point_local[b]`` (default: COM) of every body."""
    xpos, xmat, axis_w, anchor = forward_kinematics(m, q)
    nb, nv = m.nb, m.nv
    if point_local is None:
        point_local = m.body_ipos
    jacp = np.zeros((nb, 3, nv))
    jacr = np.zeros((nb, 3, nv))
    for b in range(nb):
        pt = xpos[b] + xmat[b] @ point_local[b]
        # walk up the tree
        anc = b
        chain = []
        while anc >= 0:
            chain.append(anc)
            anc = int(m.body_parent[anc])
        for j in range(nv):
            if int(m.dof_body[j]) in chain:
                if m.dof_type[j] == SLIDE:
                    jacp[b, :, j] = axis_w[j]
                else:
                    jacr[b, :, j] = axis_w[j]
                    jacp[b, :, j] = np.cross(axis_w[j], pt - anchor[j])
    return jacp, jacr, xpos, xmat


def mass_matrix(m: WalkerModel, q: np.ndarray) -> np.ndarray:
    """Joint-space inertia from body COM Jacobians (definition of kinetic energy) + armature."""
    jacp, jacr, _, xmat = body_jacobians(m, q)
    M = np.zeros((m.nv, m.nv))
    for b in range(m.nb):
        Iw = xmat[b] @ np.diag(m.body_inertia[b]) @ xmat[b].T
        M += m.body_mass[b] * jacp[b].T @ jacp[b] + jacr[b].T @ Iw @ jacr[b]
    M[np.diag_indices(m.nv)] += m.dof_armature
    return M


def _set_const(m: WalkerModel) -> None:
    """dof_invweight0 / body_invweight0 as MuJoCo's mj_setConst defines them at qpos0."""
    q0 = m.qpos0
    Minv = np.linalg.inv(mass_matrix(m, q0))
    m.dof_invweight0 = np.diag(Minv).copy()
    jacp, jacr, _, _ = body_jacobians(m, q0)
    inv = np.zeros((m.nb, 2))
    for b in range(m.nb):
        Ap = jacp[b] @ Minv @ jacp[b].T
        Ar = jacr[b] @ Minv @ jacr[b].T
        inv[b, 0] = np.trace(Ap) / 3.0
        inv[b, 1] = np.trace(Ar) / 3.0
    m.body_invweight0 = inv


# ----------------------------------------------------------------------------------------------
# builder shared by the built-in specs and the MJCF loader
# ----------------------------------------------------------------------------------------------

class _Builder:
    def __init__(self, name: str, timestep: float):
        self.name, self.timestep = name, timestep
        self.bodies: List[dict] = []
        self.dofs: List[dict] = []
        self.acts: List[dict] = []
        self.spheres: List[dict] = []
        self.boxes: List[dict] = []
        self.sites: List[dict] = []

    def body(self, name, parent, pos, mass, ipos, inertia) -> int:
        self.bodies.append(dict(name=name, parent=parent, pos=pos, mass=mass, ipos=ipos, inertia=inertia))
        return len(self.bodies) - 1

    def joint(self, name, body, jtype, axis, ref=0.0, damping=0.0, armature=0.01, limited=True,
              rng=(0.0, 0.0), pos=(0.0, 0.0, 0.0)) -> int:
        ax = np.asarray(axis, dtype=np.float64)
        k = int(np.argmax(np.abs(ax)))
        if not (abs(abs(ax[k]) - 1.0) < 1e-12 and np.count_nonzero(ax) == 1):
            raise ValueError(f"joint {name}: only +-coordinate axes are supported, got {axis}")
        if jtype == HINGE and np.any(np.asarray(pos, dtype=np.float64) != 0.0):
            raise ValueError(f"joint {name}: hinge anchors must sit at the body origin")
        self.dofs.append(dict(name=name, body=body, type=jtype, k=k, sign=float(np.sign(ax[k])), ref=ref,
                              damping=damping, armature=armature, limited=limited, rng=rng))
        return len(self.dofs) - 1

    def motor(self, joint_name, gear=1.0, ctrlrange=(-300.0, 300.0), forcerange=(-300.0, 300.0)):
        self.acts.append(dict(joint=joint_name, gear=gear, ctrlrange=ctrlrange, forcerange=forcerange))

    def capsule(self, body, fromto, radius, mu):
        a, b = np.asarray(fromto[:3], float), np.asarray(fromto[3:], float)
        # MuJoCo's plane-capsule test places one sphere at each end of the segment.
        for end in (a, b):
            self.spheres.append(dict(body=body, pos=end, radius=radius, mu=max(mu, FLOOR_FRICTION)))

    def box(self, body, pos, size, yaw, mu):
        Rb = _rot_axis(2, yaw)
        corners = np.zeros((8, 3))
        for i in range(8):           # MuJoCo corner order: bit0 -> x, bit1 -> y, bit2 -> z
            v = np.array([size[0] if i & 1 else -size[0],
                          size[1] if i & 2 else -size[1],
                          size[2] if i & 4 else -size[2]])
            corners[i] = Rb @ v
        self.boxes.append(dict(body=body, center=np.asarray(pos, float), corners=corners,
                               mu=max(mu, FLOOR_FRICTION)))

    def site(self, body, pos):
        self.sites.append(dict(body=body, pos=np.asarray(pos, float)))

    def finish(self) -> WalkerModel:
        B, D, A = self.bodies, self.dofs, self.acts
        names = [d["name"] for d in D]
        f64 = np.float64
        m = WalkerModel(
            name=self.name, timestep=self.timestep,
            body_names=[b["name"] for b in B],
            body_parent=np.array([b["parent"] for b in B], np.int32),
            body_pos=np.array([b["pos"] for b in B], f64),
            body_mass=np.array([b["mass"] for b in B], f64),
            body_ipos=np.array([b["ipos"] for b in B], f64),
            body_inertia=np.array([b["inertia"] for b in B], f64),
            dof_names=names,
            dof_body=np.array([d["body"] for d in D], np.int32),
            dof_type=np.array([d["type"] for d in D], np.int32),
            dof_axis_idx=np.array([d["k"] for d in D], np.int32),
            dof_axis_sign=np.array([d["sign"] for d in D], f64),
            dof_ref=np.array([d["ref"] for d in D], f64),
            dof_damping=np.array([d["damping"] for d in D], f64),
            dof_armature=np.array([d["armature"] for d in D], f64),
            dof_limited=np.array([1 if d["limited"] else 0 for d in D], np.uint8),
            dof_range=np.array([d["rng"] for d in D], f64),
            act_names=[a["joint"] for a in A],
            act_dof=np.array([names.index(a["joint"]) for a in A], np.int32),
            act_gear=np.array([a["gear"] for a in A], f64),
            act_ctrlrange=np.array([a["ctrlrange"] for a in A], f64),
            act_forcerange=np.array([a["forcerange"] for a in A], f64),
            sphere_body=np.array([s["body"] for s in self.spheres], np.int32),
            sphere_pos=np.array([s["pos"] for s in self.spheres], f64).reshape(-1, 3),
            sphere_radius=np.array([s["radius"] for s in self.spheres], f64),
            sphere_mu=np.array([s["mu"] for s in self.spheres], f64),
            box_body=np.array([b["body"] for b in self.boxes], np.int32),
            box_center=np.array([b["center"] for b in self.boxes], f64).reshape(-1, 3),
            box_corner=np.array([b["corners"] for b in self.boxes], f64).reshape(-1, 8, 3),
            box_mu=np.array([b["mu"] for b in self.boxes], f64),
            site_body=np.array([s["body"] for s in self.sites], np.int32),
            site_pos=np.array([s["pos"] for s in self.sites], f64).reshape(-1, 3),
        )
        parents = {b["parent"] for b in B}
        ee = [bx for bx in self.boxes if bx["body"] not in parents and B[bx["body"]]["parent"] >= 0
              and B[B[bx["body"]]["parent"]]["parent"] >= 0]
        m.ee_body = np.array([bx["body"] for bx in ee], np.int32)
        m.ee_pos = np.array([bx["center"] for bx in ee], f64).reshape(-1, 3)
        _set_const(m)
        return m


def _foot_sites(bld: _Builder, body: int, left: bool):
    # reference: walker3d_flat_feet.xml:39-42 (right), :61-64 (left); identical in walker_165cm_65kg.xml:49-52,72-75
    y_fl, y_fr = (0.06, -0.04) if left else (0.04, -0.06)
    bld.site(body, (0.1775, y_fl, -0.08))
    bld.site(body, (0.1775, y_fr, -0.08))
    bld.site(body, (-0.0425, 0.05, -0.08))
    bld.site(body, (-0.0425, -0.05, -0.08))


def walker3d() -> WalkerModel:
    """StraightMimicWalker: 14 DoF, 8 motors (reference: drloco/mujoco/xml/walker3d_flat_feet.xml)."""
    b = _Builder("walker3d", 0.001)                                        # xml:11
    torso = b.body("torso", -1, (0, 0, 1.08), 53.5, (0, 0, 0.35), (2.5, 4.0, 1.5))   # xml:15-16
    root = dict(damping=0.0, armature=0.0, limited=False)
    b.joint("com_x", torso, SLIDE, (1, 0, 0), **root)                      # xml:18
    b.joint("com_y", torso, SLIDE, (0, 1, 0), **root)                      # xml:19
    b.joint("com_z", torso, SLIDE, (0, 0, 1), ref=1.08, pos=(0, 0, -1.08), **root)   # xml:20
    b.joint("trunk_rot_x", torso, HINGE, (1, 0, 0), **root)                # xml:21
    b.joint("trunk_rot_y", torso, HINGE, (0, 1, 0), **root)                # xml:22
    b.joint("trunk_rot_z", torso, HINGE, (0, 0, 1), **root)                # xml:23
    b.capsule(torso, (0, 0, 0, 0, 0, 0.7), 0.075, 0.9)                     # xml:25
    for side, y, front_rng, yaw in (("right", -0.08, (-0.7854, 0.0873), -0.05),
                                    ("left", 0.08, (-0.0873, 0.7854), 0.05)):   # xml:26-46 / 48-68
        left = side == "left"
        thigh = b.body(f"thigh_{side}", torso, (0, y, 0), 8.5, (0, 0, -0.2), (0.15, 0.15, 0.03))
        b.joint(f"hip_sagittal_{side}", thigh, HINGE, (0, 1, 0), damping=28, rng=(-0.8727, 0.8727))
        b.joint(f"hip_frontal_{side}", thigh, HINGE, (1, 0, 0), damping=28, rng=front_rng)
        b.capsule(thigh, (0, 0, -0.05, 0, 0, -0.45), 0.05, 0.9)
        shank = b.body(f"shank_{side}", thigh, (0, 0, -0.5), 3.5, (0, 0, -0.2), (0.05, 0.05, 0.003))
        b.joint(f"knee_{side}", shank, HINGE, (0, 1, 0), damping=12, rng=(0.0, 2.6180))
        b.capsule(shank, (0, 0, -0.05, 0, 0, -0.45), 0.04, 0.9)
        foot = b.body(f"foot_{side}", shank, (0, 0, -0.5), 1.5, (0.06, 0, -0.07), (0.003, 0.006, 0.005))
        b.joint(f"ankle_{side}", foot, HINGE, (0, 1, 0), damping=20, rng=(-0.3491, 0.6981))
        b.box(foot, (0.0675, 0.005 if left else -0.005, -0.04), (0.11, 0.05, 0.04), yaw, 0.9)
        _foot_sites(b, foot, left)
    for j in ("hip_sagittal_right", "hip_frontal_right", "knee_right", "ankle_right",
              "hip_sagittal_left", "hip_frontal_left", "knee_left", "ankle_left"):   # xml:71-80
        b.motor(j)
    return b.finish()


def walker165() -> WalkerModel:
    """MimicWalker165cm65kg: 19 DoF, 13 motors (reference: drloco/mujoco/xml/walker_165cm_65kg.xml)."""
    b = _Builder("walker_165cm_65kg", 0.001)                               # xml:11
    pelvis = b.body("pelvis", -1, (0, 0, 1.035), 10.87, (0, 0, 0), (0.51, 0.82, 0.31))   # xml:15-18
    root = dict(damping=0.0, armature=0.0, limited=False)
    b.joint("pelvis_tx", pelvis, SLIDE, (1, 0, 0), **root)                 # xml:21
    b.joint("pelvis_tz", pelvis, SLIDE, (0, -1, 0), **root)                # xml:22
    b.joint("pelvis_ty", pelvis, SLIDE, (0, 0, 1), ref=1.035, **root)      # xml:23
    b.joint("pelvis_list", pelvis, HINGE, (1, 0, 0), **root)               # xml:24
    b.joint("pelvis_tilt", pelvis, HINGE, (0, -1, 0), **root)              # xml:25
    b.joint("pelvis_rotation", pelvis, HINGE, (0, 0, 1), **root)           # xml:26
    b.box(pelvis, (0, 0, 0.05), (0.05, 0.1, 0.04), 0.0, 0.9)               # xml:19
    torso = b.body("torso", pelvis, (0, 0, 0.1075), 32.5, (0, 0, 0.2475), (1.875, 3.0, 1.125))   # xml:27-28
    b.box(torso, (0, 0, 0.2475), (0.05, 0.12, 0.2475), 0.0, 0.9)           # xml:29
    lum = dict(damping=0.0, armature=0.0)
    b.joint("lumbar_bending", torso, HINGE, (1, 0, 0), rng=(-0.2, 0.15), **lum)      # xml:30
    b.joint("lumbar_extension", torso, HINGE, (0, -1, 0), rng=(-0.15, 0.15), **lum)  # xml:31
    b.joint("lumbar_rotation", torso, HINGE, (0, 0, 1), rng=(-0.15, 0.15), **lum)    # xml:32
    for s, y, add_axis, shank_end, ankle_axis, ankle_rng, yaw in (
            ("r", -0.08, (1, 0, 0), -0.4272, (0, 1, 0), (-0.3491, 0.6981), -0.05),    # xml:34-55
            ("l", 0.08, (-1, 0, 0), -0.45, (0, -1, 0), (-0.6981, 0.3491), 0.05)):     # xml:57-78 (Q25)
        left = s == "l"
        thigh = b.body(f"thigh_{s}", pelvis, (0, y, 0), 6.9, (0, 0, -0.2136), (0.122, 0.122, 0.024))
        b.joint(f"hip_flexion_{s}", thigh, HINGE, (0, -1, 0), damping=28, rng=(-0.8727, 0.8727))
        b.joint(f"hip_adduction_{s}", thigh, HINGE, add_axis, damping=28, rng=(-0.7854, 0.0873))
        b.joint(f"hip_rotation_{s}", thigh, HINGE, (0, 0, -1), damping=28, rng=(-0.26, 0.26))
        b.capsule(thigh, (0, 0, -0.05, 0, 0, -0.4272), 0.05, 0.9)
        shank = b.body(f"shank_{s}", thigh, (0, 0, -0.4772), 2.8, (0, 0, -0.2136), (0.04, 0.04, 0.0024))
        b.joint(f"knee_angle_{s}", shank, HINGE, (0, -1, 0), damping=12, rng=(-2.6180, 0.0))
        b.capsule(shank, (0, 0, -0.05, 0, 0, shank_end), 0.04, 0.9)
        foot = b.body(f"foot_{s}", shank, (0, 0, -0.4772), 1.2, (0.06, 0, -0.07), (0.003, 0.006, 0.005))
        b.joint(f"ankle_angle_{s}", foot, HINGE, ankle_axis, damping=20, rng=ankle_rng)
        b.box(foot, (0.0675, 0.005 if left else -0.005, -0.04), (0.11, 0.05, 0.04), yaw, 0.9)
        _foot_sites(b, foot, left)
    for j in ("lumbar_extension", "lumbar_bending", "lumbar_rotation",     # xml:82-94 (actuator order != joint order)
              "hip_flexion_r", "hip_adduction_r", "hip_rotation_r", "knee_angle_r", "ankle_angle_r",
              "hip_flexion_l", "hip_adduction_l", "hip_rotation_l", "knee_angle_l", "ankle_angle_l"):
        b.motor(j)
    return b.finish()


_BUILTIN = {"StraightMimicWalker": walker3d, "MimicWalker165cm65kg": walker165}
_CACHE: Dict[str, WalkerModel] = {}


def get_model(env_id: str) -> WalkerModel:
    """env id -> compiled model (ids as in reference drloco/mujoco/config.py:5-10)."""
    if env_id not in _BUILTIN:
        raise KeyError(f"unknown env id {env_id!r}; expected one of {sorted(_BUILTIN)}")
    if env_id not in _CACHE:
        _CACHE[env_id] = _BUILTIN[env_id]()
    return _CACHE[env_id]


# ----------------------------------------------------------------------------------------------
# MJCF subset loader
# ----------------------------------------------------------------------------------------------

def _floats(s: Optional[str], default: Sequence[float]) -> Tuple[float, ...]:
    return tuple(float(x) for x in s.split()) if s is not None else tuple(default)


def load_mjcf(path: str) -> WalkerModel:
    """Parse the MJCF subset the reference walkers use (single default class, local coordinates, radians)."""
    root = ET.parse(path).getroot()
    comp = root.find("compiler")
    if comp is not None:
        if comp.get("angle", "degree") != "radian" or comp.get("coordinate", "local") != "local":
            raise ValueError("only angle=radian, coordinate=local MJCF is supported")
        if comp.get("inertiafromgeom", "auto") != "false":
            raise ValueError("only inertiafromgeom=false MJCF is supported")
    dflt = root.find("default")
    dj = dflt.find("joint").attrib if dflt is not None and dflt.find("joint") is not None else {}
    dm = dflt.find("motor").attrib if dflt is not None and dflt.find("motor") is not None else {}
    dg = dflt.find("geom").attrib if dflt is not None and dflt.find("geom") is not None else {}
    opt = root.find("option")
    if opt is None or opt.get("integrator", "Euler") != "RK4":
        raise ValueError("reference walkers use integrator=RK4")
    bld = _Builder(root.get("model", "walker"), float(opt.get("timestep", "0.002")))

    def geom_mu(g) -> float:
        return _floats(g.get("friction", dg.get("friction")), (1.0,))[0]

    def visit(elem, parent: int):
        inert = elem.find("inertial")
        if inert is None:
            raise ValueError(f"body {elem.get('name')}: explicit <inertial> required")
        idx = bld.body(elem.get("name"), parent, _floats(elem.get("pos"), (0, 0, 0)), float(inert.get("mass")),
                       _floats(inert.get("pos"), (0, 0, 0)), _floats(inert.get("diaginertia"), (0, 0, 0)))
        for j in elem.findall("joint"):
            att = dict(dj)
            att.update(j.attrib)
            jt = {"slide": SLIDE, "hinge": HINGE}[att.get("type", "hinge")]
            limited = att.get("limited", "false") == "true"
            bld.joint(att["name"], idx, jt, _floats(att.get("axis"), (0, 0, 1)), ref=float(att.get("ref", 0)),
                      damping=float(att.get("damping", 0)), armature=float(att.get("armature", 0)),
                      limited=limited, rng=_floats(att.get("range"), (0, 0)),
                      pos=(0, 0, 0) if jt == SLIDE else _floats(att.get("pos"), (0, 0, 0)))
        for g in elem.findall("geom"):
            gt = g.get("type", dg.get("type", "sphere"))
            if gt == "capsule":
                bld.capsule(idx, _floats(g.get("fromto"), ()), _floats(g.get("size"), ())[0], geom_mu(g))
            elif gt == "box":
                aa = _floats(g.get("axisangle"), (0, 0, 1, 0))
                if aa[0] != 0 or aa[1] != 0:
                    raise ValueError("box geoms may only be yawed about z")
                bld.box(idx, _floats(g.get("pos"), (0, 0, 0)), _floats(g.get("size"), ()), aa[3] * np.sign(aa[2]),
                        geom_mu(g))
            else:
                raise ValueError(f"unsupported geom type {gt}")
        for s in elem.findall("site"):
            bld.site(idx, _floats(s.get("pos"), (0, 0, 0)))
        for child in elem.findall("body"):
            visit(child, idx)

    for top in root.find("worldbody").findall("body"):
        visit(top, -1)
    for mot in root.find("actuator").findall("motor"):
        att = dict(dm)
        att.update(mot.attrib)
        big = (-1e30, 1e30)
        bld.motor(att["joint"], float(att.get("gear", "1").split()[0]),
                  _floats(att.get("ctrlrange"), big) if att.get("ctrllimited") == "true" else big,
                  _floats(att.get("forcerange"), big) if att.get("forcelimited") == "true" else big)
    # canonical dof names differ between the built-in spec and the file; the motors were resolved by name above
    return bld.finish()
