"""Opt-in DeepMimic contact termination (EnvConfig(contact_termination=True), drl_set_contact_termination).

With the option on, an episode also ends when a body that carries none of the foot-corner sites (every body but the
two feet) touches the floor: one of its contact candidates (a box corner, or a capsule end sphere at centre_z - radius)
is at or below z = 0.  The check runs once per control step, at the state the step ends in; a blow-up wins and
playback skips it.  The step is terminal like a fall (reward -0, +0 with the timeout), and a per-env counter of such
episodes is served as get_attr("contact_terminations").

The CPU reference of the rule is defined here, on top of the pinned oracle (oracle/env_oracle.py restates the
reference, which has no such rule): the body frames come from the oracle's own float64 kinematics (body COM and xmat
of oracle/walker_physics.c), not from drloco_b200.model.forward_kinematics."""
import ctypes as C
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
KNEES = {W3D: ((8, 12), 1.0), W165: ((12, 17), -1.0)}      # knee dofs and the sign that flexes them


# --------------------------------------------------------------------------------------------------------------------
# CPU reference of the rule
# --------------------------------------------------------------------------------------------------------------------
def body_frames(phys, q):
    """float64 body origins and rotations in the world frame: origin = COM - xmat @ ipos"""
    com, xmat = phys.body_com(np.asarray(q, np.float64))
    return com - np.einsum("bij,bj->bi", xmat, phys.model.body_ipos), xmat


def candidate_heights(m, origin, xmat):
    """(body, lowest z) of every floor-contact candidate: the 8 corners of every box, every capsule end sphere"""
    bodies, z = [], []
    for k, b in enumerate(m.box_body):
        z.extend(origin[b, 2] + (m.box_center[k] + m.box_corner[k]) @ xmat[b, 2])
        bodies += [int(b)] * 8
    for s, b in enumerate(m.sphere_body):
        z.append(origin[b, 2] + xmat[b, 2] @ m.sphere_pos[s] - m.sphere_radius[s])
        bodies.append(int(b))
    return np.array(bodies), np.array(z)


def clearance(m, origin, xmat, mask):
    """lowest candidate height over the bodies of mask; the rule: touching <=> clearance <= 0"""
    b, z = candidate_heights(m, origin, xmat)
    return float(z[((mask >> b) & 1).astype(bool)].min())


class _Frames:
    """the oracle's kinematics (body frames, sites) for physics objects that do not serve them"""

    def __init__(self, model):
        from oracle.physics import OraclePhysics
        self._p = OraclePhysics(model)
        self.model = model

    def body_com(self, q):
        return self._p.body_com(q)


class ContactOracleEnv(OracleMimicEnv):
    """OracleMimicEnv whose step also ends the episode when a listed body touches the floor at the step's end state"""

    def __init__(self, spec, physics, mask):
        super().__init__(spec, physics)
        self.mask = mask
        self.kin = _Frames(spec.model)
        self.contact = False
        self.clearance = np.inf
        self.contact_terminations = 0

    def step(self, action):
        prev = (self.pos_rew, self.vel_rew, self.com_rew)
        obs, reward, done, info = super().step(action)
        self.contact = False
        if info.get("blowup") or self._PLAYBACK_REF_TRAJECS:
            return obs, reward, done, info
        self.clearance = clearance(self.spec.model, *body_frames(self.kin, self.qpos), self.mask)
        self.contact = self.clearance <= 0.0
        if self.contact:
            self.contact_terminations += 1
            if not done:                       # a terminal step: the imitation terms keep the previous step's values
                self.pos_rew, self.vel_rew, self.com_rew = prev
                done, reward = True, self._get_ET_reward()
        return obs, reward, done, info


class ContactOracleVecEnv(OracleVecEnv):
    def __init__(self, spec, n_envs, make_physics):
        self.spec, self.num_envs = spec, n_envs
        mask = M.contact_body_mask(spec.model)
        self.envs = [OracleMonitor(ContactOracleEnv(spec, make_physics(), mask)) for _ in range(n_envs)]


class _FrozenPhysics:
    """'no physics': states are injected; sites come from the oracle's kinematics"""

    def __init__(self, model):
        from oracle.physics import OraclePhysics
        self._p = OraclePhysics(model)
        self.qacc_warm = self._p.qacc_warm

    def step(self, q, v, ctrl, nsub):
        return False

    def site_xpos(self, q):
        return self._p.site_xpos(q)


def _spec(env_id, **kw):
    return make_spec(EnvConfig(env_id=env_id, **kw))


# --------------------------------------------------------------------------------------------------------------------
# CPU: which bodies, the geometry of the rule, RSI states
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("env_id,mask", [(W3D, 0x37), (W165, 0x6F)])
def test_listed_bodies_are_all_but_the_feet(env_id, mask):
    m = M.get_model(env_id)
    assert M.contact_body_mask(m) == mask
    listed = [m.body_names[b] for b in range(m.nb) if (mask >> b) & 1]
    assert not any(n.startswith("foot") for n in listed) and len(listed) == m.nb - 2
    assert sorted(set(m.site_body.tolist())) == sorted(b for b in range(m.nb) if not (mask >> b) & 1)


@pytest.mark.parametrize("env_id", [W3D, W165])
def test_qpos0_does_not_touch(env_id):
    m = M.get_model(env_id)
    kin = _Frames(m)
    c = clearance(m, *body_frames(kin, m.qpos0), M.contact_body_mask(m))
    assert c > 0.05
    # the feet stand on the floor: every candidate, feet included, is at or above the lowest foot-corner site
    _, z = candidate_heights(m, *body_frames(kin, m.qpos0))
    assert z.min() > -1e-12


@pytest.mark.parametrize("env_id", [W3D, W165])
def test_lowered_root_with_flexed_knees_puts_a_shank_sphere_below_the_floor(env_id):
    """kneeling: both knees flexed (W3D 1.6 rad, W165 1.2 rad) and the root lowered (0.55 m, 0.45 m; still above
    fall_z); the lowest listed candidate is then a shank sphere, below the floor.  The same knees without the lowering
    touch nothing."""
    m = M.get_model(env_id)
    kin = _Frames(m)
    mask = M.contact_body_mask(m)
    knees, sign = KNEES[env_id]
    shanks = [int(m.dof_body[j]) for j in knees]
    assert all(m.body_names[b].startswith("shank") for b in shanks)
    q = m.qpos0.copy()
    flex, lower = {W3D: (1.6, 0.55), W165: (1.2, 0.45)}[env_id]
    q[list(knees)] += sign * flex
    assert clearance(m, *body_frames(kin, q), mask) > 0.0
    q[2] -= lower
    assert q[2] > EnvConfig().fall_z
    b, z = candidate_heights(m, *body_frames(kin, q))
    listed = ((mask >> b) & 1).astype(bool)
    k = int(np.argmin(np.where(listed, z, np.inf)))
    assert b[k] in shanks and k >= 8 * len(m.box_body)                 # a sphere (after the box corners)
    assert z[k] < 0.0 and clearance(m, *body_frames(kin, q), mask) == z[k]


def test_zero_distance_counts_as_touching():
    """a capsule end sphere whose lowest point is exactly at z = 0 touches; one ulp higher it does not (a copy of the
    W3D model whose lower right-shank sphere has dyadic dimensions, so that the heights are exact)"""
    import copy
    m = copy.deepcopy(M.get_model(W3D))
    mask = M.contact_body_mask(m)
    s = int(np.nonzero(m.sphere_body == 2)[0][-1])                     # lower end of the right shank
    m.sphere_pos[s] = (0.0, 0.0, -0.25)
    m.sphere_radius[s] = 0.25
    xmat = np.broadcast_to(np.eye(3), (m.nb, 3, 3)).copy()
    origin = np.zeros((m.nb, 3))
    origin[:, 2] = 10.0
    origin[2, 2] = 0.5
    assert clearance(m, origin, xmat, mask) == 0.0
    origin[2, 2] = np.nextafter(0.5, 1.0)
    assert clearance(m, origin, xmat, mask) > 0.0
    origin[2, 2] = np.nextafter(0.5, 0.0)
    assert clearance(m, origin, xmat, mask) < 0.0


@pytest.mark.parametrize("env_id", [W3D, W165])
def test_no_rsi_state_touches(env_id):
    """every sample of the mocap, after the RSI ground shift, keeps every listed body above the floor"""
    from oracle.physics import OraclePhysics
    spec = _spec(env_id)
    m, t = spec.model, spec.mocap
    env = ContactOracleEnv(spec, OraclePhysics(m), M.contact_body_mask(m))
    lowest = np.inf
    n = 0
    for i in range(t.n_steps):
        for pos in range(int(t.step_len[i])):
            env.reset(i, pos)
            # reset() already took the cursor's first step; the state is the RSI state
            c = clearance(m, *body_frames(env.kin, env.qpos), env.mask)
            lowest = min(lowest, c)
            n += 1
    assert n == sum(int(x) for x in t.step_len)
    # the smallest clearance is 9.03 cm on W3D (lower shank sphere) and 6.74 cm on W165 (lower shank sphere)
    assert lowest > {W3D: 0.09, W165: 0.067}[env_id], lowest


def test_config_default_is_off():
    assert EnvConfig().contact_termination is False
    assert EnvConfig(contact_termination=True).contact_termination is True


@pytest.fixture(scope="module")
def built_lib():
    if not os.path.exists(lib.LIB_PATH):
        sys.path.insert(0, REPO)
        import __graft_entry__
        __graft_entry__.build()
    return lib.load()


def test_abi_argument_errors_without_a_device(built_lib):
    assert built_lib.drl_set_contact_termination(None, 0x37) == -1             # DRL_ERR_INVALID
    assert b"null env" in built_lib.drl_last_error()
    out = (C.c_int32 * 4)()
    assert built_lib.drl_get_contact_terminations(None, C.cast(out, C.c_void_p), None) == -1
    assert b"null argument" in built_lib.drl_last_error()


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
    """done, reward sign, observations, terminal observations, cursors, Monitor values and the counter against the
    oracle on injected states (frame_skip = 0): perturbed states, some kneeling with a shank below the floor above
    fall_z, some below fall_z.  States whose listed clearance is within 1 mm of the floor are lifted by 2 mm, so that
    float32 and float64 kinematics cannot disagree on the answer."""
    n, steps = 32, 60
    env = _gpu_env(env_id, n, ep_dur_max=25, contact_termination=True)
    spec = env.spec
    m = spec.model
    mask = M.contact_body_mask(m)
    kin = _Frames(m)
    (k_r, k_l), sign = KNEES[env_id]
    env.debug_set(frame_skip_override=0)
    ora = ContactOracleVecEnv(spec, n, lambda: _FrozenPhysics(m))
    if eval_mode:
        env.env_method("activate_evaluation")
        for e in ora.envs:
            e.env._EVAL_MODEL = True
    rng = np.random.default_rng(3)
    istep, pos = _rsi(spec, n, rng)
    og, oo = env.reset(inject=(istep, pos)), ora.reset(istep, pos)
    assert _rel(og, oo) < 2e-5
    np.testing.assert_array_equal(env.get_attr("contact_terminations"), 0)
    n_done = n_contact = n_contact_above_fall = 0
    for k in range(steps):
        qg, vg, cg = env.get_state()
        q_new = qg + (0.02 * rng.standard_normal(qg.shape)).astype(np.float32)
        v_new = vg + (0.2 * rng.standard_normal(vg.shape)).astype(np.float32)
        u = rng.random(n)
        fall, kneel = u < 0.03, (u >= 0.03) & (u < 0.13)
        q_new[fall, 2] = 0.45
        for i in np.nonzero(kneel)[0]:
            q_new[i, 2] -= rng.uniform(0.35, 0.6)
            q_new[i, k_r if rng.random() < 0.5 else k_l] += sign * rng.uniform(1.0, 2.0)
        for i in range(n):
            if abs(clearance(m, *body_frames(kin, q_new[i].astype(np.float64)), mask)) < 1e-3:
                q_new[i, 2] += np.float32(2e-3)
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
        np.testing.assert_array_equal(env.get_attr("contact_terminations"),
                                      [e.env.contact_terminations for e in ora.envs])
        np.testing.assert_array_equal(env.get_state()[2], _ora_state(ora)[2])
        contact = np.array([e.env.contact for e in ora.envs])
        n_done += int(do.sum())
        n_contact += int(contact.sum())
        n_contact_above_fall += int((contact & (q_new[:, 2] >= spec.cfg.fall_z)).sum())
    assert n_done > 20 and n_contact > 10 and n_contact_above_fall > 5
    for name in ("mean_ep_pos_rew_smoothed", "mean_ep_com_rew_smoothed", "mean_reward_smoothed", "ep_ret_smoothed",
                 "ep_len_smoothed"):
        got = np.array(env.get_attr(name))
        want = np.array([float(getattr(e, name)) for e in ora.envs])
        np.testing.assert_allclose(got, want, rtol=2e-4, atol=2e-5, err_msg=name)
    rec = env.episode_records()
    want_et = [p for e in ora.envs for p in e.et_positions]
    assert sorted(rec["et_pos"].tolist()) == sorted(want_et)
    env.close()


def _unmirror_tables(spec):
    oi, osn, _, _ = spec.mirror_tables()
    oi, osn = np.asarray(oi), np.asarray(osn, np.float64)
    return oi, osn


def _q_from_obs(spec, obs, left):
    """the joint configuration of an (optionally mirrored) observation, com_x = 0"""
    m = spec.model
    o = np.asarray(obs, np.float64)
    if left:
        oi, osn = _unmirror_tables(spec)
        u = np.empty_like(o)
        u[oi] = o * osn                     # obs_mirrored[k] = sign[k] * obs[idx[k]]
        o = u
    head = spec.obs_dim - (m.nv - 1) - m.nv
    return np.r_[0.0, o[head:head + m.nv - 1]]


def _left_after_next(spec, cursor):
    """is the step the cursor moves to at the next control step a left step? (stepwise cursor, random RSI)"""
    t = spec.mocap
    i, p = int(cursor[0]), int(cursor[1])
    if p + t.increment - int(t.step_len[i]) + 1 > 0:
        i = (0 if t.left_step[i] else 1) if i >= t.n_steps - 1 else i + 1
    return bool(t.left_step[i])


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,integrator", [(W3D, "rk4"), (W3D, "euler"), (W165, "rk4")])
def test_random_action_rollouts_respect_the_rule(env_id, integrator):
    """full physics, random actions, several hundred steps: no env that goes on has a listed body more than 1e-4 below
    the floor; every counted episode ended with one at most 1e-4 above it (its terminal observation, un-mirrored, in
    the CPU rule), and every other terminal state that is not a timeout keeps them above -1e-4"""
    n, steps, margin = 256, 300, 1e-4
    env = _gpu_env(env_id, n, seed=11, integrator=integrator, contact_termination=True)
    spec = env.spec
    m = spec.model
    mask = M.contact_body_mask(m)
    kin = _Frames(m)
    rng = np.random.default_rng(7)
    env.reset()
    counts = np.zeros(n, np.int64)
    n_counted = 0
    for k in range(steps):
        cur = env.get_state()[2]
        a = rng.uniform(-1, 1, (n, env.act_dim)).astype(np.float32)
        _, _, d, info = env.step(a)
        q = env.get_state()[0]
        new_counts = np.array(env.get_attr("contact_terminations"))
        inc = new_counts - counts
        assert ((inc == 0) | ((inc == 1) & d)).all(), k
        counts = new_counts
        for i in range(n):
            if not d[i]:
                assert clearance(m, *body_frames(kin, q[i].astype(np.float64)), mask) > -margin, (k, i)
                continue
            left = spec.mirror and _left_after_next(spec, cur[i])
            qt = _q_from_obs(spec, info[i]["terminal_observation"], left)
            c = clearance(m, *body_frames(kin, qt), mask)
            if inc[i]:
                n_counted += 1
                assert c <= margin, (k, i, c)
            elif int(cur[i, 3]) + 1 < spec.cfg.ep_dur_max and qt[2] >= spec.cfg.fall_z:
                assert c > -margin, (k, i, c)
    assert n_counted > 0
    st = env.stats()
    assert st["blowups"] == 0
    assert int(counts.sum()) == n_counted
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,steps", [(W3D, 8), (W165, 6)])
def test_rollout_parity_short_horizon_with_the_rule(env_id, steps):
    """full physics (RK4) with the rule on; the same contact-sensitivity exclusion and 1e-4 bar as the rollout test
    without it"""
    from oracle.sensitivity import SensitivityProbe
    n = 64
    env = _gpu_env(env_id, n, contact_termination=True)
    spec = env.spec
    probes = []

    def make():
        probes.append(SensitivityProbe(spec.model, cabi.INTEGRATOR_RK4, seed=len(probes)))
        return probes[-1]
    ora = ContactOracleVecEnv(spec, n, make)
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
        rows = np.maximum(np.maximum(_rel_rows(qg, qo), _rel_rows(vg, vo)), np.abs(rg - ro))
        ok = ~flagged
        np.testing.assert_array_equal(dg[ok], do[ok], err_msg=f"done flags, step {k}")
        np.testing.assert_array_equal(cg[ok], co[ok], err_msg=f"cursor, step {k}")
        cnt_g = np.array(env.get_attr("contact_terminations"))
        cnt_o = np.array([e.env.contact_terminations for e in ora.envs])
        np.testing.assert_array_equal(cnt_g[ok], cnt_o[ok], err_msg=f"counter, step {k}")
        assert rows[ok].max() < 1e-4, (k, np.nonzero(rows >= 1e-4)[0], np.nonzero(flagged)[0], rows.max())
    assert int(np.array([p.flagged for p in probes]).sum()) <= n // 5
    env.close()


def _run_tensor(env, acts, at=None):
    """reset + steps on the tensor path; every output of the run.  at: {step index: callable(env)} run before that
    step"""
    import torch
    outs = [env.reset_tensor().clone()]
    for k, a in enumerate(acts):
        if at and k in at:
            at[k](env)
        o, r, d = env.step_tensor(a)
        outs += [o.clone(), r.clone(), d.clone()]
    q, v, c = env.get_state()
    return dict(outs=torch.cat([x.float().flatten() for x in outs]).cpu().numpy(), q=q, v=v, c=c,
                stats=env.stats(), extras=env.extras().cpu().numpy(), ring=env.episode_records())


def _assert_runs_equal(a, b):
    for k in ("outs", "q", "v", "c", "extras"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert a["stats"] == b["stats"]
    # the episode ring: slots are taken in the order in which thread blocks finish, so compare the records as a set
    rec = lambda r: sorted(zip(*(r[k].tolist() for k in sorted(r))))   # noqa: E731
    assert rec(a["ring"]) == rec(b["ring"])


def _set_mask(mask):
    def f(env):
        lib.check(lib.load().drl_set_contact_termination(env._handle, mask), "drl_set_contact_termination")
    return f


@pytest.mark.gpu
def test_switching_on_then_off_restores_the_outputs():
    """on -> mask 0, before the first step and in the middle of a run, gives every output of an env that never
    enabled it, bit for bit; the run with the rule on ends more episodes"""
    import torch
    from drloco_b200.vec_env import B200MimicVecEnv
    n, steps, mid = 256, 250, 100
    g = torch.Generator(device="cuda")
    g.manual_seed(4)
    acts = torch.rand(steps, n, 8, device="cuda", generator=g) * 2 - 1
    cfg = EnvConfig(env_id=W3D)
    mask = M.contact_body_mask(M.get_model(W3D))

    def run(at=None, before=None, c=cfg):
        env = B200MimicVecEnv(W3D, num_envs=n, cfg=c, seed=9)
        for f in before or ():
            f(env)
        out = _run_tensor(env, acts, at)
        env.close()
        return out
    fresh = run()
    on, off = _set_mask(mask), _set_mask(0)
    _assert_runs_equal(run(before=[on, off]), fresh)
    _assert_runs_equal(run(at={mid: lambda e: (on(e), off(e))}), fresh)
    with_rule = run(c=EnvConfig(env_id=W3D, contact_termination=True))
    assert with_rule["stats"]["episodes"] > fresh["stats"]["episodes"]


@pytest.mark.gpu
def test_call_order_and_argument_errors():
    import torch
    l = lib.load()
    env = _gpu_env(W3D, 8)                                            # rule off (default)
    env.reset()
    out = torch.zeros(8, dtype=torch.int32, device="cuda")
    assert l.drl_get_contact_terminations(env._handle, C.c_void_p(out.data_ptr()), None) == -3   # DRL_ERR_STATE
    assert b"never enabled" in l.drl_last_error()
    with pytest.raises(AttributeError):
        env.get_attr("contact_terminations")
    env.close()
    spec = make_spec()
    cfg = cabi.DrlConfig()
    cfg.num_envs, cfg.device, cfg.frame_skip, cfg.obs_dim, cfg.act_dim, cfg.ctrl_freq = 8, 0, 5, 29, 8, 200.0
    h = C.c_void_p()
    assert l.drl_create(C.byref(cfg), C.byref(h)) == 0
    assert l.drl_set_contact_termination(h, 0x37) == -3                 # DRL_ERR_STATE: no model yet
    assert b"upload the model" in l.drl_last_error()
    cm = cabi.pack_model(spec.model)
    assert l.drl_upload_model(h, C.byref(cm)) == 0
    for bad in (1 << 7, 0x80000000, 0x37 | (1 << 3), 1 << 6, 0x7F):    # a bit >= nb; a foot (carries the sites)
        assert l.drl_set_contact_termination(h, bad) == -1, hex(bad)     # DRL_ERR_INVALID
    assert l.drl_get_contact_terminations(h, C.c_void_p(out.data_ptr()), None) == -3
    assert l.drl_set_contact_termination(h, 0) == 0                     # off stays off: no counter yet
    assert l.drl_get_contact_terminations(h, C.c_void_p(out.data_ptr()), None) == -3
    assert l.drl_set_contact_termination(h, 0x37) == 0
    assert l.drl_get_contact_terminations(h, C.c_void_p(out.data_ptr()), None) == 0
    assert l.drl_get_contact_terminations(h, None, None) == -1
    torch.cuda.synchronize()
    assert out.cpu().tolist() == [0] * 8
    assert l.drl_destroy(h) == 0


@pytest.mark.gpu
def test_vecnormalize_graph_path_equals_the_tensor_path():
    import torch
    from drloco_b200.vec_env import B200VecNormalize
    n, steps = 256, 250
    rng = np.random.default_rng(6)
    acts = rng.uniform(-1, 1, (steps, n, 8)).astype(np.float32)
    res, counts = [], []
    for graph in (True, False):
        env = _gpu_env(W3D, n, seed=13, contact_termination=True)
        vn = B200VecNormalize(env)
        outs = []
        if graph:
            vn.reset()
            for a in acts:
                o, r, d, _ = vn.step(a)
                outs.append((np.array(o), np.array(r), np.array(d)))
            assert vn.use_graph and getattr(vn, "_graphs", None)            # the captured path ran
        else:
            vn.reset_tensor()
            for a in acts:
                o, r, d = vn.step_tensor(torch.from_numpy(a).cuda())
                outs.append((o.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy().astype(bool)))
        res.append(outs)
        counts.append(env.get_attr("contact_terminations"))
        env.close()
    assert any(d.any() for _, _, d in res[0]) and sum(counts[0]) > 0
    assert counts[0] == counts[1]
    for (o1, r1, d1), (o2, r2, d2) in zip(*res):
        np.testing.assert_array_equal(o1, o2)
        np.testing.assert_array_equal(r1, r2)
        np.testing.assert_array_equal(d1, d2)


@pytest.mark.gpu
def test_two_identical_runs_are_bit_identical():
    import torch
    n, steps = 512, 250
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    acts = torch.rand(steps, n, 8, device="cuda", generator=g) * 2 - 1
    runs, counts = [], []
    for _ in range(2):
        env = _gpu_env(W3D, n, seed=21, contact_termination=True)
        runs.append(_run_tensor(env, acts))
        counts.append(env.get_attr("contact_terminations"))
        env.close()
    _assert_runs_equal(*runs)
    assert counts[0] == counts[1] and sum(counts[0]) > 0
