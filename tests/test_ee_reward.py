"""The optional DeepMimic end-effector (foot position) reward term (EnvConfig.ee_weight / ee_scale).

ee_rew = exp(-ee_scale * S), S = sum over the model's end-effector points (the foot-box centres) of the squared distance
between the simulated point and the point of the reference pose at the cursor, both relative to the root-body origin in
world axes.  The reward becomes (w_pos*pos + w_vel*vel + w_com*com + ee_weight*ee_rew) * rew_scale + alive_bonus.

The CPU reference of the term is defined here, on top of the pinned oracle (oracle/env_oracle.py restates the
reference, which has no such term): the points come from the oracle's own float64 kinematics (body COM and xmat of
oracle/walker_physics.c), not from drloco_b200.model.forward_kinematics, so the check does not share code with the
product's kinematics."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest

from drloco_b200 import cabi, lib
from drloco_b200 import model as M
from drloco_b200.config import EnvConfig
from drloco_b200.walkers import make_spec
from oracle.env_oracle import OracleMimicEnv, OracleMonitor, OracleVecEnv

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W3D, W165 = "StraightMimicWalker", "MimicWalker165cm65kg"


# --------------------------------------------------------------------------------------------------------------------
# CPU reference of the term
# --------------------------------------------------------------------------------------------------------------------
class EEOracleEnv(OracleMimicEnv):
    """OracleMimicEnv whose imitation reward has the end-effector term (needs ``physics.body_com``)."""

    def __init__(self, spec, physics):
        super().__init__(spec, physics)
        self.ee_rew = 0.0
        self.ee_sq_err = 0.0

    def ee_positions(self, q):
        """end-effector points relative to the root-body origin, world axes: body origin = COM - xmat @ ipos"""
        m = self.spec.model
        com, xmat = self.phys.body_com(np.asarray(q, np.float64))
        origin = com - np.einsum("bij,bj->bi", xmat, m.body_ipos)
        pts = origin[m.ee_body] + np.einsum("eij,ej->ei", xmat[m.ee_body], m.ee_pos)
        return pts - origin[0]

    def get_ee_reward(self):
        dif = self.ee_positions(self.qpos) - self.ee_positions(self.refs.get_qpos())
        self.ee_sq_err = float(np.sum(np.square(dif)))
        return float(np.exp(-self.cfg.ee_scale * self.ee_sq_err))

    def get_imitation_reward(self):
        w_pos, w_vel, w_com, _ = self.cfg.rew_weights
        self.pos_rew, self.vel_rew, self.com_rew = self.get_pose_reward(), self.get_vel_reward(), self.get_com_reward()
        self.ee_rew = self.get_ee_reward()
        return (w_pos * self.pos_rew + w_vel * self.vel_rew + w_com * self.com_rew
                + self.cfg.ee_weight * self.ee_rew) * self.cfg.rew_scale


class EEOracleMonitor(OracleMonitor):
    """OracleMonitor with the per-step list of ee_rew (never cleared, like the other components) and its smoothed
    mean at every episode end."""

    def __init__(self, env):
        super().__init__(env)
        self.ep_ee_rews = []
        self.mean_ep_ee_rew_smoothed = 0

    def step(self, action):
        obs, reward, done, info = super().step(action)
        self.ep_ee_rews.append(self.env.ee_rew)
        if done:
            self.mean_ep_ee_rew_smoothed = self._smooth("ep_ee_rew", float(np.mean(self.ep_ee_rews)))
        return obs, reward, done, info


class EEOracleVecEnv(OracleVecEnv):
    def __init__(self, spec, n_envs, make_physics):
        self.spec, self.num_envs = spec, n_envs
        self.envs = [EEOracleMonitor(EEOracleEnv(spec, make_physics())) for _ in range(n_envs)]


class _FrozenPhysics:
    """'no physics': states are injected; sites and body frames come from the oracle's kinematics."""

    def __init__(self, model):
        from oracle.physics import OraclePhysics
        self._p = OraclePhysics(model)
        self.qacc_warm = self._p.qacc_warm

    def step(self, q, v, ctrl, nsub):
        return False

    def site_xpos(self, q):
        return self._p.site_xpos(q)

    def body_com(self, q):
        return self._p.body_com(q)


def _spec(env_id, **kw):
    return make_spec(EnvConfig(env_id=env_id, **kw))


def _cpu_env(env_id, **kw):
    from oracle.physics import OraclePhysics
    spec = _spec(env_id, **kw)
    return EEOracleEnv(spec, OraclePhysics(spec.model))


class _FixedRef:
    """cursor stand-in whose reference pose is a given qpos"""

    def __init__(self, q):
        self.q = np.array(q, np.float64)

    def get_qpos(self):
        return self.q.copy()


# --------------------------------------------------------------------------------------------------------------------
# CPU: model data and the term's definition
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("env_id", [W3D, W165])
def test_end_effectors_are_the_two_foot_box_centres(env_id):
    m = M.get_model(env_id)
    assert m.ee_body.dtype == np.int32 and m.ee_pos.shape == (2, 3)
    assert sorted(m.body_names[b] for b in m.ee_body) == sorted(n for n in m.body_names if n.startswith("foot"))
    for b, p in zip(m.ee_body, m.ee_pos):
        assert not (m.body_parent == b).any()                  # a leaf
        (k,) = np.nonzero(m.box_body == b)[0]
        np.testing.assert_array_equal(p, m.box_center[k])
    cm = cabi.pack_model(m)
    assert cm.n_ee == 2 and list(cm.ee_body)[:2] == list(m.ee_body)
    np.testing.assert_array_equal(np.ctypeslib.as_array(cm.ee_pos)[:2], m.ee_pos)


def test_known_answer_knee_rotation():
    """W3D at qpos0: every body frame is aligned with the world, the knee axis is world y.  Bending one knee by d moves
    that foot-box centre on a circle about the knee axis: a chord of 2 r sin(d/2), r = the distance of the centre from
    the axis in the sagittal (x-z) plane, read off the model tables by hand."""
    env = _cpu_env(W3D, ee_weight=0.3)
    m = env.spec.model
    j = m.dof_names.index("knee_right")
    foot = m.body_names.index("foot_right")
    assert tuple(m.dof_axis_idx[j:j + 1]) == (1,) and m.dof_axis_sign[j] == 1.0
    (e,) = np.nonzero(m.ee_body == foot)[0]
    knee_to_centre = m.body_pos[foot] + m.ee_pos[e]                 # the shank origin is the knee
    r = math.hypot(knee_to_centre[0], knee_to_centre[2])
    for d in (0.05, 0.3, -0.7):
        env.refs = _FixedRef(m.qpos0)
        env.qpos = m.qpos0.copy()
        env.qpos[j] += d
        got = env.get_ee_reward()
        want = math.exp(-40.0 * (2 * r * math.sin(d / 2)) ** 2)
        assert abs(got - want) <= 1e-12, (d, got, want)
        assert abs(env.ee_sq_err - (2 * r * math.sin(d / 2)) ** 2) <= 1e-14


@pytest.mark.parametrize("env_id", [W3D, W165])
def test_rsi_gives_ee_reward_one(env_id):
    """reference-state initialisation copies the reference pose: zero error, ee_rew = 1 (and the reference's post-RSI
    check, imitation reward > 0.95 rew_scale, holds with the term on)"""
    env = _cpu_env(env_id, ee_weight=0.3)
    t = env.spec.mocap
    rng = np.random.default_rng(0)
    for _ in range(200):
        i = int(rng.integers(0, t.n_steps))
        env.reset(i, int(rng.integers(0, t.step_len[i])))
        assert abs(env.ee_rew - 1.0) <= 1e-12 and env.ee_sq_err <= 1e-24


@pytest.mark.parametrize("env_id", [W3D, W165])
def test_root_translation_leaves_ee_reward_unchanged(env_id):
    env = _cpu_env(env_id, ee_weight=0.3)
    m, t = env.spec.model, env.spec.mocap
    rng = np.random.default_rng(1)
    for row in rng.integers(0, t.n_samples, 20):
        ref = t.ref[row, :m.nv].copy()
        q = ref + 0.1 * rng.standard_normal(m.nv)
        env.refs = _FixedRef(ref)
        env.qpos = q.copy()
        base = env.get_ee_reward()
        assert 0.0 < base < 1.0
        for shift in ([5.0, -2.0, 0.3], [-40.0, 3.0, -0.6]):
            env.qpos = q.copy()
            env.qpos[:3] += shift                                   # the three root slides
            assert abs(env.get_ee_reward() - base) <= 1e-12


def test_defaults_leave_the_term_off():
    """ee_weight = 0 keeps the reference's reward; ee_scale defaults to DeepMimic's coefficient"""
    c = EnvConfig()
    assert c.ee_weight == 0.0 and c.ee_scale == 40.0


# --------------------------------------------------------------------------------------------------------------------
# CPU: C ABI layout and argument checks that run before any device is touched
# --------------------------------------------------------------------------------------------------------------------
def test_abi_v4_keeps_the_ee_fields_appended(tmp_path):
    import subprocess
    probe = tmp_path / "probe.c"
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "drloco_b200.h"\n'
                     'int main(void){printf("%d %d %zu %zu %zu %zu %zu\\n", DRL_ABI_VERSION, DRL_MAX_EE,'
                     ' offsetof(DrlWalkerModel, n_ee), offsetof(DrlWalkerModel, ee_body),'
                     ' offsetof(DrlWalkerModel, ee_pos), offsetof(DrlConfig, ee_weight), offsetof(DrlConfig, ee_scale));'
                     'return 0;}\n')
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(REPO, "include"), str(probe), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    W, Cf = cabi.DrlWalkerModel, cabi.DrlConfig
    assert got == [cabi.DRL_ABI_VERSION, cabi.MAX_EE, W.n_ee.offset, W.ee_body.offset, W.ee_pos.offset,
                   Cf.ee_weight.offset, Cf.ee_scale.offset]
    assert cabi.DRL_ABI_VERSION == 4
    # appended: every field of the previous layout keeps its offset
    assert W.n_ee.offset > W.site_pos.offset and Cf.ee_weight.offset > Cf.monitor_median_torque.offset


@pytest.fixture(scope="module")
def built_lib():
    if not os.path.exists(lib.LIB_PATH):
        sys.path.insert(0, REPO)
        import __graft_entry__
        __graft_entry__.build()
    return lib.load()


@pytest.mark.parametrize("weight,scale", [(-0.1, 40.0), (float("nan"), 40.0), (float("inf"), 40.0), (0.3, 0.0),
                                          (0.3, -1.0), (0.3, float("nan"))])
def test_create_rejects_bad_ee_config(built_lib, weight, scale):
    cfg = cabi.DrlConfig()
    cfg.num_envs, cfg.device, cfg.frame_skip, cfg.obs_dim, cfg.act_dim, cfg.ctrl_freq = 8, 0, 5, 29, 8, 200.0
    cfg.ee_weight, cfg.ee_scale = weight, scale
    h = C.c_void_p()
    assert built_lib.drl_create(C.byref(cfg), C.byref(h)) == -1                 # DRL_ERR_INVALID
    assert b"ee_" in built_lib.drl_last_error()


# --------------------------------------------------------------------------------------------------------------------
# GPU
# --------------------------------------------------------------------------------------------------------------------
def _gpu_env(env_id, n, **kw):
    from drloco_b200.vec_env import B200MimicVecEnv
    seed = kw.pop("seed", 5)
    return B200MimicVecEnv(env_id, num_envs=n, cfg=EnvConfig(env_id=env_id, **kw), seed=seed)


def _rsi(spec, n, rng):
    t = spec.mocap
    istep = rng.integers(0, t.n_steps, n).astype(np.int32)
    pos = np.array([rng.integers(0, t.step_len[i]) for i in istep], np.int32)
    return istep, pos


def _rel_rows(x, ref):
    scale = np.maximum(1.0, np.abs(ref).max(axis=-1, keepdims=True))
    return (np.abs(x - ref) / scale).max(axis=-1)


def _rel(x, ref):
    return float(_rel_rows(x, ref).max())


def _ora_state(ora):
    q = np.stack([e.env.qpos for e in ora.envs])
    v = np.stack([e.env.qvel for e in ora.envs])
    c = np.array([[e.env.refs.i_step, e.env.refs.pos, e.env.refs.count_steps_same_vel, e.env.ep_dur] for e in ora.envs])
    return q, v, c


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,eval_mode", [(W3D, False), (W165, False), (W3D, True)])
def test_env_logic_and_monitor_on_injected_states(env_id, eval_mode):
    """reward, termination, cursor and Monitor statistics with the term on, on injected states (frame_skip = 0): W3D
    (stepwise cursor, mirrored policy), W165 (wrap cursor) and W3D in evaluation mode (deterministic inits, whose
    reference rows come from step 0's table until the first step transition)"""
    n, steps = 32, 60
    env = _gpu_env(env_id, n, ep_dur_max=25, ee_weight=0.3)
    spec = env.spec
    env.debug_set(frame_skip_override=0)
    ora = EEOracleVecEnv(spec, n, lambda: _FrozenPhysics(spec.model))
    if eval_mode:
        env.env_method("activate_evaluation")
        for m in ora.envs:
            m.env._EVAL_MODEL = True
    rng = np.random.default_rng(3)
    istep, pos = _rsi(spec, n, rng)
    og, oo = env.reset(inject=(istep, pos)), ora.reset(istep, pos)
    assert _rel(og, oo) < 2e-5
    np.testing.assert_array_equal(env.get_attr("ee_rew"), 1.0)
    n_done, ee_seen = 0, []
    for k in range(steps):
        qg, vg, cg = env.get_state()
        dq = (0.02 * rng.standard_normal(qg.shape)).astype(np.float32)
        dv = (0.2 * rng.standard_normal(vg.shape)).astype(np.float32)
        q_new, v_new = qg + dq, vg + dv
        fall = rng.random(n) < 0.03
        q_new[fall, 2] = 0.45
        env.set_state(q_new, v_new, cg)
        for i, e in enumerate(ora.envs):
            e.env.qpos[:] = q_new[i].astype(np.float64)
            e.env.qvel[:] = v_new[i].astype(np.float64)
        a = rng.uniform(-1.5, 1.5, (n, env.act_dim)).astype(np.float32)
        og, rg, dg, ig = env.step(a, inject=(istep, pos))
        oo, ro, do, io = ora.step(a, istep, pos)
        np.testing.assert_array_equal(dg, do)
        np.testing.assert_array_equal(np.signbit(rg), np.signbit(ro))
        assert np.abs(rg - ro).max() < 2e-5
        assert _rel(og, oo) < 2e-5
        for i in np.nonzero(do)[0]:
            assert _rel(ig[i]["terminal_observation"][None], io[i]["terminal_observation"][None]) < 2e-5
        ee_g = np.array(env.get_attr("ee_rew"))
        ee_o = np.array([m.env.ee_rew for m in ora.envs])
        assert np.abs(ee_g - ee_o).max() < 2e-5, k
        ee_seen.append(ee_o[~do])
        np.testing.assert_array_equal(env.get_state()[2], _ora_state(ora)[2])
        n_done += int(do.sum())
    assert n_done > 20
    ee_seen = np.concatenate(ee_seen)
    assert ee_seen.min() < 0.9 and ee_seen.max() < 1.0             # the term is exercised, not saturated at 1
    for name in ("mean_ep_ee_rew_smoothed", "mean_ep_pos_rew_smoothed", "mean_reward_smoothed", "ep_ret_smoothed"):
        got = np.array(env.get_attr(name))
        want = np.array([float(getattr(m, name)) for m in ora.envs])
        np.testing.assert_allclose(got, want, rtol=2e-4, atol=2e-5, err_msg=name)
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", [W3D, W165])
def test_ee_error_geometry(env_id):
    """ee_scale = 1 and 0.2 rad perturbations: -log(ee_rew) against the oracle's S, 1e-4 relative - the geometry, not a
    saturated exponential"""
    n = 64
    env = _gpu_env(env_id, n, ee_weight=0.3, ee_scale=1.0)
    spec = env.spec
    env.debug_set(frame_skip_override=0)
    ora = EEOracleVecEnv(spec, n, lambda: _FrozenPhysics(spec.model))
    rng = np.random.default_rng(4)
    istep, pos = _rsi(spec, n, rng)
    env.reset(inject=(istep, pos))
    ora.reset(istep, pos)
    qg, vg, cg = env.get_state()
    q_new = qg.copy()
    q_new[:, 3:] += (0.2 * rng.standard_normal((n, spec.model.nv - 3))).astype(np.float32)
    env.set_state(q_new, vg, cg)
    for i, e in enumerate(ora.envs):
        e.env.qpos[:] = q_new[i].astype(np.float64)
        e.env.qvel[:] = vg[i].astype(np.float64)
    a = np.zeros((n, env.act_dim), np.float32)
    _, _, dg, _ = env.step(a, inject=(istep, pos))
    _, _, do, _ = ora.step(a, istep, pos)
    ok = ~(dg | do)
    assert ok.sum() >= n - 4
    s_gpu = -np.log(np.array(env.get_attr("ee_rew"), np.float64))
    s_ora = np.array([m.env.ee_sq_err for m in ora.envs])
    assert (s_ora[ok] > 1e-3).all()
    rel = np.abs(s_gpu[ok] - s_ora[ok]) / s_ora[ok]
    assert rel.max() < 1e-4, rel.max()
    env.close()


class _ProbeWithFrames:
    """contact-sensitivity probe (oracle/sensitivity.py) that also serves body frames"""

    def __new__(cls, model, integ, seed):
        from oracle.sensitivity import SensitivityProbe
        p = SensitivityProbe(model, integ, seed=seed)
        p.body_com = p._p.body_com
        return p


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,steps", [(W3D, 8), (W165, 6)])
def test_rollout_parity_short_horizon_with_term(env_id, steps):
    """full physics (RK4) with the term on; the same contact-sensitivity exclusion and 1e-4 bar as the rollout test
    without it"""
    n = 64
    env = _gpu_env(env_id, n, ee_weight=0.3)
    spec = env.spec
    probes = []

    def make():
        probes.append(_ProbeWithFrames(spec.model, cabi.INTEGRATOR_RK4, len(probes)))
        return probes[-1]
    ora = EEOracleVecEnv(spec, n, make)
    rng = np.random.default_rng(1)
    istep, pos = _rsi(spec, n, rng)
    og, oo = env.reset(inject=(istep, pos)), ora.reset(istep, pos)
    assert _rel(og, oo) < 2e-5
    for k in range(steps):
        a = rng.uniform(-1, 1, (n, spec.act_dim)).astype(np.float32)
        og, rg, dg, _ = env.step(a, inject=(istep, pos))
        oo, ro, do, _ = ora.step(a, istep, pos)
        qg, vg, cg = env.get_state()
        qo, vo, co = _ora_state(ora)
        for i in np.nonzero(do & dg)[0]:
            probes[i].clear()
        flagged = np.array([p.flagged for p in probes])
        ee_g = np.array(env.get_attr("ee_rew"))
        ee_o = np.array([m.env.ee_rew for m in ora.envs])
        rows = np.maximum(np.maximum(_rel_rows(qg, qo), _rel_rows(vg, vo)), np.abs(rg - ro))
        rows = np.maximum(rows, np.abs(ee_g - ee_o))
        ok = ~flagged
        np.testing.assert_array_equal(dg[ok], do[ok], err_msg=f"done flags, step {k}")
        np.testing.assert_array_equal(cg[ok], co[ok], err_msg=f"cursor, step {k}")
        assert rows[ok].max() < 1e-4, (k, np.nonzero(rows >= 1e-4)[0], np.nonzero(flagged)[0], rows.max())
    assert int(np.array([p.flagged for p in probes]).sum()) <= n // 5
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", [W3D, W165])
def test_playback_earns_the_maximum_reward(env_id):
    n, T = 8, 200
    env = _gpu_env(env_id, n, ee_weight=0.3)
    rng = np.random.default_rng(2)
    istep, pos = _rsi(env.spec, n, rng)
    env.set_playback(True)
    env.reset(inject=(istep, pos))
    c = env.cfg
    want = c.rew_scale * (sum(c.rew_weights[:3]) + c.ee_weight) + c.alive_bonus
    a = np.zeros((n, env.act_dim), np.float32)
    for _ in range(T):
        _, r, d, _ = env.step(a, inject=(istep, pos))
        assert not d.any()
        assert np.abs(r - want).max() < 1e-6
        np.testing.assert_array_equal(env.get_attr("ee_rew"), 1.0)
    env.close()


@pytest.mark.gpu
def test_call_order_and_argument_errors():
    import torch
    l = lib.load()
    env = _gpu_env(W3D, 8)                                            # term off (default)
    env.reset()
    out = torch.zeros(8, device="cuda")
    p = C.c_void_p(out.data_ptr())
    assert l.drl_get_ee_reward(env._handle, p, p, None) == -3          # DRL_ERR_STATE
    assert b"ee_weight" in l.drl_last_error()
    for name in ("ee_rew", "mean_ep_ee_rew_smoothed"):
        with pytest.raises(AttributeError):
            env.get_attr(name)
    env.close()
    spec = make_spec()
    cfg = cabi.DrlConfig()
    cfg.num_envs, cfg.device, cfg.frame_skip, cfg.obs_dim, cfg.act_dim, cfg.ctrl_freq = 8, 0, 5, 29, 8, 200.0
    cfg.ee_weight, cfg.ee_scale = 0.3, 40.0
    for field, value in (("n_ee", 0), ("n_ee", 5), ("n_ee", -1), ("ee_body", 7)):
        h = C.c_void_p()
        assert l.drl_create(C.byref(cfg), C.byref(h)) == 0
        cm = cabi.pack_model(spec.model)
        if field == "n_ee":
            cm.n_ee = value
        else:
            cm.ee_body[1] = value
        assert l.drl_upload_model(h, C.byref(cm)) == -1, (field, value)   # DRL_ERR_INVALID
        assert l.drl_destroy(h) == 0
    # the term off accepts a model without points
    cfg.ee_weight = 0.0
    h = C.c_void_p()
    assert l.drl_create(C.byref(cfg), C.byref(h)) == 0
    cm = cabi.pack_model(spec.model)
    cm.n_ee = 0
    assert l.drl_upload_model(h, C.byref(cm)) == 0
    assert l.drl_destroy(h) == 0


@pytest.mark.gpu
def test_two_identical_runs_are_bit_identical():
    import torch
    n, steps = 512, 40
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    acts = torch.rand(steps, n, 8, device="cuda", generator=g) * 3 - 1.5
    runs = []
    for _ in range(2):
        env = _gpu_env(W3D, n, seed=21, ep_dur_max=15, ee_weight=0.3)
        env.reset_tensor()
        rews = []
        for k in range(steps):
            _, r, _ = env.step_tensor(acts[k])
            rews.append(r.clone())
        names = ("ee_rew", "mean_ep_ee_rew_smoothed", "mean_ep_pos_rew_smoothed", "ep_ret_smoothed")
        runs.append(dict(stats=env.stats(), attrs={k: env.get_attr(k) for k in names}, rews=torch.stack(rews)))
        env.close()
    a, b = runs
    assert a["stats"] == b["stats"] and a["stats"]["episodes"] > 0
    assert a["attrs"] == b["attrs"]
    assert torch.equal(a["rews"], b["rews"])
