"""Model compiler (drloco_b200/model.py): built-in walker specs vs the reference MJCF files, compile-time constants."""
import dataclasses
import os

import numpy as np
import pytest

from drloco_b200 import model as M

# the reference's own MJCF files, in the verbatim copy of its `drloco` package that baseline/build_ref.py makes
REF_XML = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                       "baseline", "_ref", "drloco", "mujoco", "xml", "")


@pytest.mark.parametrize("env_id,xml,nv,nu,nb,mass", [
    ("StraightMimicWalker", "walker3d_flat_feet.xml", 14, 8, 7, 80.5),
    ("MimicWalker165cm65kg", "walker_165cm_65kg.xml", 19, 13, 8, 65.17)])
def test_builtin_specs(env_id, xml, nv, nu, nb, mass):
    m = M.get_model(env_id)
    assert (m.nv, m.nu, m.nb) == (nv, nu, nb)
    assert abs(m.total_mass - mass) < 1e-9                     # SURVEY.md §8a (a4)
    assert np.all(m.act_ctrlrange == [-300, 300]) and np.all(m.act_forcerange == [-300, 300])
    assert len(m.site_body) == 8
    if os.path.exists(REF_XML + xml):                          # only where the reference copy was made
        ref = M.load_mjcf(REF_XML + xml)
        for f in dataclasses.fields(m):
            x, y = getattr(m, f.name), getattr(ref, f.name)
            if isinstance(x, np.ndarray):
                np.testing.assert_array_equal(x, y, err_msg=f.name)


def test_w3d_structure():
    m = M.get_model("StraightMimicWalker")
    # motors follow qpos order 6..13 (xml:71-80); root joints unlimited and without armature
    assert list(m.act_dof) == list(range(6, 14))
    assert not m.dof_limited[:6].any() and m.dof_limited[6:].all()
    assert np.all(m.dof_armature[:6] == 0) and np.all(m.dof_armature[6:] == 0.01)
    assert m.dof_ref[2] == 1.08 and m.qpos0[2] == 1.08
    # at qpos0 every foot-corner site touches the ground plane exactly
    xpos, xmat, _, _ = M.forward_kinematics(m, m.qpos0)
    z = [xpos[b][2] + (xmat[b] @ p)[2] for b, p in zip(m.site_body, m.site_pos)]
    np.testing.assert_allclose(z, 0.0, atol=1e-12)


def test_w165_actuator_order():
    m = M.get_model("MimicWalker165cm65kg")
    names = [m.dof_names[j] for j in m.act_dof]
    assert names[:3] == ["lumbar_extension", "lumbar_bending", "lumbar_rotation"]      # Q25
    # left shank capsule is longer than the right one (xml:66 vs :43)
    ends = m.sphere_pos[:, 2]
    assert -0.45 in ends and -0.4272 in ends


def test_invweight_constants():
    """dof_invweight0 = diag(M^-1) and body_invweight0 = mean diag of J M^-1 J' at qpos0 (MuJoCo mj_setConst)."""
    m = M.get_model("StraightMimicWalker")
    Minv = np.linalg.inv(M.mass_matrix(m, m.qpos0))
    np.testing.assert_allclose(m.dof_invweight0, np.diag(Minv), rtol=1e-12)
    # a free-floating 80.5 kg system: translational inverse weight of the root is bounded below by 1/total mass
    assert m.body_invweight0[0, 0] >= 1.0 / m.total_mass - 1e-12
    assert np.all(m.body_invweight0 > 0)
    # left / right symmetry
    np.testing.assert_allclose(m.body_invweight0[1:4], m.body_invweight0[4:7], rtol=1e-9)


def test_unsupported_models_are_rejected():
    b = M._Builder("bad", 0.001)
    t = b.body("torso", -1, (0, 0, 1), 1.0, (0, 0, 0), (1, 1, 1))
    with pytest.raises(ValueError):
        b.joint("skew", t, M.HINGE, (0.6, 0.8, 0))
    with pytest.raises(ValueError):
        b.joint("offset", t, M.HINGE, (1, 0, 0), pos=(0, 0, 0.1))
