"""Opt-in PD position-servo actuation (EnvConfig(actuation="pd", pd_kp=..., pd_kv=...), drl_set_actuation).

Every motor becomes a MuJoCo <position kp kv> servo: the clipped action a_u maps to the target ctrl_u = mid_u + a_u half_u
over the range of the joint it drives (float32), the policy mirror applies after the map, and at every dynamics
evaluation f_u = clamp(kp_u (ctrl_u - gear_u q) - kv_u gear_u v, forcerange_u), tau = gear_u f_u, from that evaluation's
q and v.  The Monitor torque is mean |f| at the state the step starts from.

The CPU reference is defined here on top of the pinned oracle, which stays as it is: one PD evaluation is the oracle's
motor evaluation (oracle/walker_physics.c, orc_forward) with ctrl set to the servo force computed at that evaluation's
state - exact, because both walkers' force range lies inside their ctrlrange - and the integrators restate the
oracle's RK4 / semi-implicit Euler loops around it, recording the same constraint-set signatures for the
contact-sensitivity probe (oracle/sensitivity.py)."""
import copy
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
from oracle.env_oracle import OracleMimicEnv, OracleVecEnv, OracleMonitor

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W3D, W165 = "StraightMimicWalker", "MimicWalker165cm65kg"
# test gains, well inside the explicit-RK4 stability estimate of the ankle (h (kv + damping) / I < 2.8 at 1 ms)
KP, KV = 200.0, 5.0


# --------------------------------------------------------------------------------------------------------------------
# CPU reference of the servo
# --------------------------------------------------------------------------------------------------------------------
def servo_force(m, kp, kv, q, v, ctrl):
    """actuator forces f [nu] of the servos at (q, v) for the targets ctrl (float64)"""
    j, g = m.act_dof, m.act_gear
    cc = np.minimum(m.dof_range[j, 1], np.maximum(m.dof_range[j, 0], ctrl))
    f = kp * (cc - g * q[j]) - kv * (g * v[j])
    return np.minimum(m.act_forcerange[:, 1], np.maximum(m.act_forcerange[:, 0], f))


class PDOraclePhysics:
    """OraclePhysics-compatible float64 physics with PD servos: every evaluation is the oracle's orc_forward with ctrl
    set to the servo force at that evaluation's state; RK4 and Euler as oracle/walker_physics.c step_sig."""

    def __init__(self, model, integrator, kp, kv):
        from oracle.physics import OraclePhysics, lib as olib
        # the motor path of the oracle clamps ctrl to ctrlrange, then to forcerange: a force inside forcerange passes
        # unchanged when forcerange lies inside ctrlrange
        assert (model.act_ctrlrange[:, 0] <= model.act_forcerange[:, 0]).all()
        assert (model.act_ctrlrange[:, 1] >= model.act_forcerange[:, 1]).all()
        self.model, self.integrator = model, integrator
        self.kp = np.broadcast_to(np.asarray(kp, np.float64), (model.nu,)).copy()
        self.kv = np.broadcast_to(np.asarray(kv, np.float64), (model.nu,)).copy()
        self._p = OraclePhysics(model, integrator)
        self._l = olib()
        self.cm = self._p.cm
        self.qacc_warm = self._p.qacc_warm
        self.nv = model.nv

    def force(self, q, v, ctrl):
        return servo_force(self.model, self.kp, self.kv, np.asarray(q, np.float64), np.asarray(v, np.float64),
                           np.asarray(ctrl, np.float64))

    def _eval(self, q, v, ctrl, warm):
        """one dynamics evaluation: (qacc, (contact set, limit set)); raises on a numerical failure"""
        f = np.ascontiguousarray(self.force(q, v, ctrl))
        q, v = np.ascontiguousarray(q, np.float64), np.ascontiguousarray(v, np.float64)
        qacc = np.zeros(self.nv)
        p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
        if self._l.orc_forward(C.byref(self.cm), p(q), p(v), p(f), p(warm), p(qacc), None):
            raise FloatingPointError
        con, lim = C.c_ulonglong(), C.c_ulonglong()
        self._l.orc_get_last_sets(C.byref(con), C.byref(lim))
        return qacc, (con.value, lim.value)

    def forward(self, q, v, ctrl):
        return self._eval(q, v, ctrl, np.zeros(self.nv))[0]

    @staticmethod
    def _blown(q, v):
        return not (np.isfinite(q).all() and np.isfinite(v).all() and np.abs(q).max() <= 1e10
                    and np.abs(v).max() <= 1e10)

    def step_trace(self, q, v, ctrl, nsub):
        """in place, like OraclePhysics.step_trace: (blew_up, uint64 [nsub, 4, 2] constraint-set signature)"""
        h, nv = self.model.timestep, self.nv
        sig = np.zeros((int(nsub), 4, 2), np.uint64)
        try:
            for s in range(int(nsub)):
                if self._blown(q, v):
                    return True, sig
                if self.integrator == cabi.INTEGRATOR_RK4:
                    A, Bw = (0.5, 0.5, 1.0), (1.0 / 6, 1.0 / 3, 1.0 / 3, 1.0 / 6)
                    kq, kvv = np.zeros((4, nv)), np.zeros((4, nv))
                    qs, vs = q.copy(), v.copy()
                    for st in range(4):
                        kvv[st], sig[s, st] = self._eval(qs, vs, ctrl, self.qacc_warm)
                        kq[st] = vs
                        if st < 3:
                            qs, vs = q + h * A[st] * kq[st], v + h * A[st] * kvv[st]
                    dq, dv = np.zeros(nv), np.zeros(nv)
                    for st in range(4):
                        dq, dv = dq + Bw[st] * kq[st], dv + Bw[st] * kvv[st]
                    q += h * dq
                    v += h * dv
                else:
                    # mj_Euler: (M + h B) a' = M a, B = joint damping only; the servo's kv is in the explicit force
                    a, sig[s, 0] = self._eval(q, v, ctrl, self.qacc_warm)
                    Mq = self._p.mass_matrix(q)
                    rhs = Mq @ a
                    Mq[np.diag_indices(nv)] += h * self.model.dof_damping
                    v += h * np.linalg.solve(Mq, rhs)
                    q += h * v
        except (FloatingPointError, np.linalg.LinAlgError):
            return True, sig
        return self._blown(q, v), sig

    def step(self, q, v, ctrl, nsub):
        return self.step_trace(q, v, ctrl, nsub)[0]

    def site_xpos(self, q):
        return self._p.site_xpos(q)


def pd_probe(model, integrator, kp, kv, seed):
    """the contact-sensitivity probe of the parity tests (oracle/sensitivity.py) stepping with the servo law"""
    from oracle.sensitivity import SensitivityProbe
    p = SensitivityProbe(model, integrator, seed=seed)
    p._p, p._probe = (PDOraclePhysics(model, integrator, kp, kv) for _ in range(2))
    p.qacc_warm = p._p.qacc_warm
    p.force = p._p.force
    return p


class PDOracleEnv(OracleMimicEnv):
    """OracleMimicEnv with the servo's action map and Monitor torque; ``physics`` must expose ``force(q, v, ctrl)``."""

    def __init__(self, spec, physics):
        super().__init__(spec, physics)
        m = spec.model
        lo, hi = m.dof_range[m.act_dof, 0], m.dof_range[m.act_dof, 1]
        self.mid, self.half = (0.5 * (lo + hi)).astype(np.float32), (0.5 * (hi - lo)).astype(np.float32)

    def _rescale_actions(self, action):
        a = np.clip(np.asarray(action, np.float32), np.float32(-1), np.float32(1))
        return self.mid + a * self.half                      # float32, like the kernel

    def step(self, action):
        q0, v0 = self.qpos.copy(), self.qvel.copy()
        out = super().step(action)                           # ctrl (the mirrored targets) -> self.last_ctrl
        self.act_force = self.phys.force(q0, v0, self.last_ctrl)
        return out


class PDOracleVecEnv(OracleVecEnv):
    def __init__(self, spec, n_envs, make_physics):
        self.spec, self.num_envs = spec, n_envs
        self.envs = [OracleMonitor(PDOracleEnv(spec, make_physics())) for _ in range(n_envs)]


class _FrozenPD:
    """'no physics' (states are injected), with the servo force and the oracle's sites"""

    def __init__(self, model, kp, kv):
        self._p = PDOraclePhysics(model, cabi.INTEGRATOR_RK4, kp, kv)
        self.qacc_warm = self._p.qacc_warm
        self.force = self._p.force

    def step(self, q, v, ctrl, nsub):
        return False

    def site_xpos(self, q):
        return self._p.site_xpos(q)


def _free_model(env_id):
    """the walker without joint damping and joint limits (the servo law alone acts on the joints)"""
    m = copy.deepcopy(M.get_model(env_id))
    m.dof_damping[:] = 0
    m.dof_limited[:] = 0
    return m


# --------------------------------------------------------------------------------------------------------------------
# CPU: the reference's evaluation, mechanics and action map
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("env_id", [W3D, W165])
@pytest.mark.parametrize("kp", [KP, 4000.0])
def test_one_evaluation_is_the_servo_force_through_the_motor_path(env_id, kp):
    """in free flight (no contact, no limit row) the PD evaluation's qacc is M^-1 (sum_u e_j(u) gear_u f_u - D v - c)
    with M, c from the oracle and f from the servo law; kp = 4000 drives most servos into the force clamp"""
    m = M.get_model(env_id)
    P = PDOraclePhysics(_free_model(env_id), cabi.INTEGRATOR_RK4, kp, 3.0)
    rng = np.random.default_rng(0)
    clamped = 0
    for _ in range(5):
        q = m.qpos0 + 0.3 * rng.standard_normal(m.nv)
        q[2] = 4.0
        v = rng.standard_normal(m.nv)
        u = rng.uniform(-1, 1, m.nu)
        lo, hi = m.dof_range[m.act_dof, 0], m.dof_range[m.act_dof, 1]
        ctrl = 0.5 * (lo + hi) + u * 0.5 * (hi - lo)
        f = kp * (ctrl - m.act_gear * q[m.act_dof]) - 3.0 * (m.act_gear * v[m.act_dof])
        clamped += int((np.abs(f) > 300.0).sum())
        f = np.clip(f, -300.0, 300.0)
        tau = np.zeros(m.nv)
        tau[m.act_dof] = m.act_gear * f
        want = np.linalg.solve(P._p.mass_matrix(q), tau - P._p.bias(q, v))
        got, sets = P._eval(q, v, ctrl, np.zeros(m.nv))
        assert sets == (0, 0)
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-9 * max(1.0, np.abs(want).max()))
        np.testing.assert_array_equal(P.force(q, v, ctrl), f)
        # and the motor path with ctrl = f is the same evaluation, bit for bit
        np.testing.assert_array_equal(got, P._p.forward(q, v, f)[0])
    assert clamped < 5 * m.nu and (clamped > 0 or kp < 1000.0)       # kp = 4000: clamped and free servos both


@pytest.mark.parametrize("env_id", [W3D, W165])
def test_servo_energy_is_conserved_without_damping_and_decays_with_kv(env_id):
    """zero gravity, no joint damping or limits, lifted clear of the floor, no force clamp: with kv = 0 the energy
    1/2 v'Mv + sum_u 1/2 kp (gear q - ctrl)^2 is conserved by 200 RK4 steps to the order of the oracle's free-flight
    energy test; with kv > 0 it decreases at every step"""
    m = _free_model(env_id)
    kp = 20.0                                                       # keeps h * omega small: RK4 drift ~ (h omega)^6
    lo, hi = m.dof_range[m.act_dof, 0], m.dof_range[m.act_dof, 1]
    ctrl = 0.5 * (lo + hi)
    rng = np.random.default_rng(2)
    for kv in (0.0, 2.0):
        P = PDOraclePhysics(m, cabi.INTEGRATOR_RK4, kp, kv)
        P.cm.gravity_z = 0.0
        q = m.qpos0.copy()
        q[m.act_dof] = ctrl + 0.2 * rng.uniform(-1, 1, m.nu) * (hi - lo)
        q[2] = 6.0
        v = 0.5 * rng.standard_normal(m.nv)

        def energy(q, v):
            return 0.5 * v @ P._p.mass_matrix(q) @ v + 0.5 * np.sum(kp * (m.act_gear * q[m.act_dof] - ctrl) ** 2)
        def power(v):                                               # dissipated by the servos' kv
            return kv * np.sum((m.act_gear * v[m.act_dof]) ** 2)
        E, W = [energy(q, v)], [0.0]
        for _ in range(200):
            p0 = power(v)
            bad, sig = P.step_trace(q, v, ctrl, 1)
            assert not bad and not sig.any()
            assert np.abs(P.force(q, v, ctrl)).max() < 300.0
            E.append(energy(q, v))
            W.append(W[-1] + 0.5 * m.timestep * (p0 + power(v)))
        E = np.array(E)
        if kv == 0.0:
            assert np.abs(E - E[0]).max() < 1e-8 * E[0], np.abs(E - E[0]).max() / E[0]
        else:
            assert (np.diff(E) < 0).all() and E[-1] < 0.99 * E[0]
            # energy balance: the loss is the work of the damping term (trapezoidal rule at 1 ms)
            assert abs((E[0] - E[-1]) - W[-1]) < 1e-3 * W[-1], ((E[0] - E[-1]), W[-1])


@pytest.mark.parametrize("env_id", [W3D, W165])
def test_action_map_spans_the_joint_ranges(env_id):
    spec = make_spec(EnvConfig(env_id=env_id, actuation="pd", pd_kp=KP))
    env = PDOracleEnv(spec, _FrozenPD(spec.model, KP, 0.0))
    m = spec.model
    lo, hi = m.dof_range[m.act_dof, 0], m.dof_range[m.act_dof, 1]
    f32 = np.float32
    # to float32 rounding of mid +- half (the kernel then clamps the target to the joint range)
    for a, want in ((-1, lo), (0, 0.5 * (lo + hi)), (1, hi), (7, hi)):                  # 7: clipped to 1 first
        np.testing.assert_allclose(env._rescale_actions(np.full(m.nu, a, f32)), want, rtol=0, atol=2e-7)
    # the knee of W3D ([0, 2.618]): negative actions bend it less, they are not all mapped to 0
    t = env._rescale_actions(np.full(m.nu, -0.5, f32))
    assert ((t > lo) & (t < hi)).all()


def test_mirrored_targets_stay_in_the_mirrored_joint_range():
    spec = make_spec(EnvConfig(env_id=W3D, actuation="pd", pd_kp=KP))
    assert spec.mirror
    env = PDOracleEnv(spec, _FrozenPD(spec.model, KP, 0.0))
    m = spec.model
    lo, hi = m.dof_range[m.act_dof, 0], m.dof_range[m.act_dof, 1]
    rng = np.random.default_rng(3)
    acts = np.concatenate([rng.uniform(-1, 1, (200, m.nu)), [np.full(m.nu, -1.0), np.full(m.nu, 1.0)]])
    for a in acts.astype(np.float32):
        t = env.mirror_action(env._rescale_actions(a))
        assert ((t >= lo.astype(np.float32)) & (t <= hi.astype(np.float32))).all(), t


def test_env_config_validation():
    c = EnvConfig()
    assert c.actuation == "torque" and c.pd_kp is None and c.pd_kv is None
    kp, kv = EnvConfig(actuation="pd", pd_kp=300.0).pd_gains()
    np.testing.assert_array_equal(kp, np.full(8, 300.0))
    np.testing.assert_array_equal(kv, np.zeros(8))
    per = tuple(range(1, 14))
    kp, kv = EnvConfig(env_id=W165, actuation="pd", pd_kp=per, pd_kv=2.5).pd_gains()
    np.testing.assert_array_equal(kp, np.array(per, np.float64))
    np.testing.assert_array_equal(kv, np.full(13, 2.5))
    bad = [dict(actuation="pd"), dict(actuation="position", pd_kp=1.0), dict(pd_kp=1.0), dict(pd_kv=1.0),
           dict(actuation="pd", pd_kp=0.0), dict(actuation="pd", pd_kp=-1.0), dict(actuation="pd", pd_kp=math.inf),
           dict(actuation="pd", pd_kp=math.nan), dict(actuation="pd", pd_kp=1.0, pd_kv=-0.1),
           dict(actuation="pd", pd_kp=1.0, pd_kv=math.nan), dict(actuation="pd", pd_kp=(1.0,) * 7),
           dict(env_id=W165, actuation="pd", pd_kp=1.0, pd_kv=(1.0,) * 8)]
    for kw in bad:
        with pytest.raises(ValueError):
            EnvConfig(**kw)


@pytest.fixture(scope="module")
def built_lib():
    if not os.path.exists(lib.LIB_PATH):
        sys.path.insert(0, REPO)
        import __graft_entry__
        __graft_entry__.build()
    return lib.load()


def test_set_actuation_argument_errors_without_a_device(built_lib):
    kp = np.full(8, KP)
    p = kp.ctypes.data_as(C.c_void_p)
    for mode in (cabi.ACTUATION_TORQUE, cabi.ACTUATION_PD, 7):
        assert built_lib.drl_set_actuation(None, mode, p, p) == -1             # DRL_ERR_INVALID
        assert b"null env" in built_lib.drl_last_error()


# --------------------------------------------------------------------------------------------------------------------
# GPU
# --------------------------------------------------------------------------------------------------------------------
def _gpu_env(env_id, n, kp=KP, kv=KV, **kw):
    from drloco_b200.vec_env import B200MimicVecEnv
    seed = kw.pop("seed", 5)
    cfg = EnvConfig(env_id=env_id, actuation="pd", pd_kp=kp, pd_kv=kv, **kw)
    return B200MimicVecEnv(env_id, num_envs=n, cfg=cfg, seed=seed)


def _rsi(spec, n, rng):
    t = spec.mocap
    istep = rng.integers(0, t.n_steps, n).astype(np.int32)
    pos = np.array([rng.integers(0, t.step_len[i]) for i in istep], np.int32)
    return istep, pos


def _rel_rows(x, ref):
    scale = np.maximum(1.0, np.abs(ref).max(axis=-1, keepdims=True))
    return (np.abs(x - ref) / scale).max(axis=-1)


def _ora_state(ora):
    q = np.stack([e.env.qpos for e in ora.envs])
    v = np.stack([e.env.qvel for e in ora.envs])
    c = np.array([[e.env.refs.i_step, e.env.refs.pos, e.env.refs.count_steps_same_vel, e.env.ep_dur] for e in ora.envs])
    return q, v, c


@pytest.mark.gpu
def test_action_space_is_the_unit_box():
    env = _gpu_env(W3D, 8)
    assert env.action_space.shape == (8,)
    assert (env.action_space.low == -1).all() and (env.action_space.high == 1).all()
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,integrator,steps,kp", [(W3D, "rk4", 8, 100.0), (W3D, "euler", 8, 100.0),
                                                        (W165, "rk4", 6, 200.0)])
def test_rollout_parity_short_horizon_pd(env_id, integrator, steps, kp):
    """the criteria of the torque-mode rollout parity test: 1e-4 relative for every environment the contact-sensitivity
    probe does not flag, exact cursors and done flags there, at most 20 % flagged.

    Servos driven to random targets make more foot contacts fall within float32 resolution than random torques do, and
    the flagged fraction depends on the gain and the sample.  Measured on this sample (seed 1, 64 envs): W3D RK4 13
    flagged at kp = 200 and 9 at kp = 100; W165 RK4 16 at kp = 100 and within the bound at kp = 200 (other seeds, W3D
    RK4 at kp = 200: 19 - 34 %).  Every unflagged environment stayed below 4e-5 in all of these.  The gains here are
    the ones whose sample meets the 20 % bound; the sample is seeded and the flags come from the float64 oracle, so
    they do not vary between runs."""
    n = 64
    env = _gpu_env(env_id, n, kp=kp, integrator=integrator)
    spec = env.spec
    integ = cabi.INTEGRATOR_RK4 if integrator == "rk4" else cabi.INTEGRATOR_EULER
    probes = []

    def make():
        probes.append(pd_probe(spec.model, integ, kp, KV, len(probes)))
        return probes[-1]
    ora = PDOracleVecEnv(spec, n, make)
    rng = np.random.default_rng(1)
    istep, pos = _rsi(spec, n, rng)
    og, oo = env.reset(inject=(istep, pos)), ora.reset(istep, pos)
    assert _rel_rows(og, oo).max() < 2e-5
    moved = 0.0
    for k in range(steps):
        a = rng.uniform(-1, 1, (n, spec.act_dim)).astype(np.float32)
        q_before = env.get_state()[0]
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
        assert rows[ok].max() < 1e-4, (k, np.nonzero(rows >= 1e-4)[0], np.nonzero(flagged)[0], rows.max())
        moved = max(moved, float(np.abs(qg[~dg, 6:] - q_before[~dg, 6:]).max()))
    assert int(np.array([p.flagged for p in probes]).sum()) <= n // 5
    assert moved > 1e-3                                               # the servos do move the joints
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", [W3D, W165])
def test_monitor_torque_is_the_servo_force_at_the_start_state(env_id):
    """injected states (frame_skip = 0: the state is not integrated): mean_abs_torque, the Monitor's smoothed mean and
    median, and the abs_torque_sum statistic equal mean |f| of the servo law at the state each step starts from"""
    n, steps = 32, 40
    env = _gpu_env(env_id, n, ep_dur_max=12, median_torque=True)
    spec = env.spec
    env.debug_set(frame_skip_override=0)
    ora = PDOracleVecEnv(spec, n, lambda: _FrozenPD(spec.model, KP, KV))
    rng = np.random.default_rng(3)
    istep, pos = _rsi(spec, n, rng)
    env.reset(inject=(istep, pos))
    ora.reset(istep, pos)
    env.reset_stats()
    tor_sum, clamped = 0.0, 0
    for k in range(steps):
        qg, vg, cg = env.get_state()
        q_new = qg + (0.05 * rng.standard_normal(qg.shape)).astype(np.float32)
        v_new = vg + (2.0 * rng.standard_normal(vg.shape)).astype(np.float32)
        env.set_state(q_new, v_new, cg)
        for i, e in enumerate(ora.envs):
            e.env.qpos[:] = q_new[i].astype(np.float64)
            e.env.qvel[:] = v_new[i].astype(np.float64)
        a = rng.uniform(-1.5, 1.5, (n, env.act_dim)).astype(np.float32)
        _, _, dg, _ = env.step(a, inject=(istep, pos))
        _, _, do, _ = ora.step(a, istep, pos)
        np.testing.assert_array_equal(dg, do)
        want = np.array([m.env.get_actuator_torques(True) for m in ora.envs])
        clamped += int(sum((np.abs(m.env.act_force) >= 300.0).sum() for m in ora.envs))
        got = np.array(env.get_attr("mean_abs_torque"))
        np.testing.assert_allclose(got, want, rtol=2e-5, atol=1e-4, err_msg=f"step {k}")
        tor_sum += float(want.sum())
    assert 0 < clamped < steps * n * spec.act_dim // 2                   # both sides of the force clamp are exercised
    assert env.stats()["abs_torque_sum"] == pytest.approx(tor_sum, rel=2e-5)
    for name in ("mean_abs_ep_torque_smoothed", "median_abs_torque_smoothed"):
        got = np.array(env.get_attr(name))
        want = np.array([float(getattr(m, name)) for m in ora.envs])
        np.testing.assert_allclose(got, want, rtol=2e-5, atol=1e-4, err_msg=name)
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
                stats=env.stats(), extras=env.extras().cpu().numpy())


def _assert_runs_equal(a, b):
    for k in ("outs", "q", "v", "c", "extras"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert a["stats"] == b["stats"]


def _set(mode):
    kp, kv = np.full(8, KP), np.full(8, KV)

    def f(env):
        p = None if mode == cabi.ACTUATION_TORQUE else kp.ctypes.data_as(C.c_void_p)
        q = None if mode == cabi.ACTUATION_TORQUE else kv.ctypes.data_as(C.c_void_p)
        lib.check(lib.load().drl_set_actuation(env._handle, mode, p, q), "drl_set_actuation")
    return f


@pytest.mark.gpu
def test_switching_torque_pd_torque_restores_the_torque_outputs():
    """torque -> PD -> torque, before the first step and in the middle of a run, gives every output of a fresh torque
    env bit for bit; a step taken in between in PD mode does differ"""
    import torch
    from drloco_b200.vec_env import B200MimicVecEnv
    n, steps, mid = 256, 30, 10
    g = torch.Generator(device="cuda")
    g.manual_seed(4)
    acts = torch.rand(steps, n, 8, device="cuda", generator=g) * 3 - 1.5
    cfg = EnvConfig(env_id=W3D, ep_dur_max=20)

    def run(at=None, before=None, upto=steps):
        env = B200MimicVecEnv(W3D, num_envs=n, cfg=cfg, seed=9)
        if before:
            for f in before:
                f(env)
        out = _run_tensor(env, acts[:upto], at)
        env.close()
        return out
    fresh = run()
    pd, tq = _set(cabi.ACTUATION_PD), _set(cabi.ACTUATION_TORQUE)
    _assert_runs_equal(run(before=[pd, tq]), fresh)
    _assert_runs_equal(run(at={mid: lambda e: (pd(e), tq(e))}), fresh)
    # one PD step after `mid` torque steps: its outputs (obs, rew, done of step mid) differ from the torque run's
    D = 29
    one = run(at={mid: pd}, upto=mid + 1)
    k0 = n * D + mid * (n * D + 2 * n)
    k1 = k0 + n * D
    np.testing.assert_array_equal(one["outs"][:k0], fresh["outs"][:k0])
    assert not np.array_equal(one["outs"][k0:k1], fresh["outs"][k0:k1])


@pytest.mark.gpu
def test_call_order_and_argument_errors():
    l = lib.load()
    spec = make_spec()
    cfg = cabi.DrlConfig()
    cfg.num_envs, cfg.device, cfg.frame_skip, cfg.obs_dim, cfg.act_dim, cfg.ctrl_freq = 8, 0, 5, 29, 8, 200.0
    p = lambda x: x.ctypes.data_as(C.c_void_p)   # noqa: E731
    kp, kv = np.full(8, KP), np.full(8, KV)
    h = C.c_void_p()
    assert l.drl_create(C.byref(cfg), C.byref(h)) == 0
    assert l.drl_set_actuation(h, cabi.ACTUATION_PD, p(kp), p(kv)) == -3          # DRL_ERR_STATE: no model yet
    assert b"upload the model" in l.drl_last_error()
    cm = cabi.pack_model(spec.model)
    assert l.drl_upload_model(h, C.byref(cm)) == 0
    for mode, kp_, kv_ in ((2, kp, kv), (-1, kp, kv),
                           (cabi.ACTUATION_PD, np.r_[kp[:7], 0.0], kv), (cabi.ACTUATION_PD, np.r_[kp[:7], -5.0], kv),
                           (cabi.ACTUATION_PD, np.r_[kp[:7], np.inf], kv), (cabi.ACTUATION_PD, np.r_[kp[:7], np.nan], kv),
                           (cabi.ACTUATION_PD, kp, np.r_[kv[:7], -1.0]), (cabi.ACTUATION_PD, kp, np.r_[kv[:7], np.nan])):
        assert l.drl_set_actuation(h, mode, p(kp_), p(kv_)) == -1, (mode, kp_, kv_)   # DRL_ERR_INVALID
    assert l.drl_set_actuation(h, cabi.ACTUATION_PD, None, None) == -1
    assert l.drl_set_actuation(h, cabi.ACTUATION_PD, p(kp), p(np.zeros(8))) == 0    # kv = 0 is a valid servo
    assert l.drl_set_actuation(h, cabi.ACTUATION_TORQUE, None, None) == 0
    assert l.drl_destroy(h) == 0
    # a model whose actuated knee has no joint range
    h = C.c_void_p()
    assert l.drl_create(C.byref(cfg), C.byref(h)) == 0
    cm = cabi.pack_model(spec.model)
    cm.dof_limited[spec.model.act_dof[2]] = 0
    assert l.drl_upload_model(h, C.byref(cm)) == 0
    assert l.drl_set_actuation(h, cabi.ACTUATION_PD, p(kp), p(kv)) == -1
    assert b"joint range" in l.drl_last_error()
    assert l.drl_set_actuation(h, cabi.ACTUATION_TORQUE, None, None) == 0
    assert l.drl_destroy(h) == 0


@pytest.mark.gpu
def test_vecnormalize_graph_path_equals_the_tensor_path():
    import torch
    from drloco_b200.vec_env import B200VecNormalize
    n, steps = 256, 12
    rng = np.random.default_rng(6)
    acts = rng.uniform(-1, 1, (steps, n, 8)).astype(np.float32)
    res = []
    for graph in (True, False):
        env = _gpu_env(W3D, n, seed=13, ep_dur_max=6)
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
        env.close()
    assert any(d.any() for _, _, d in res[0])
    for (o1, r1, d1), (o2, r2, d2) in zip(*res):
        np.testing.assert_array_equal(o1, o2)
        np.testing.assert_array_equal(r1, r2)
        np.testing.assert_array_equal(d1, d2)


@pytest.mark.gpu
def test_two_identical_pd_runs_are_bit_identical():
    import torch
    n, steps = 512, 40
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    acts = torch.rand(steps, n, 8, device="cuda", generator=g) * 3 - 1.5
    runs = []
    for _ in range(2):
        env = _gpu_env(W3D, n, seed=21, ep_dur_max=15)
        runs.append(_run_tensor(env, acts))
        env.close()
    _assert_runs_equal(*runs)
    assert runs[0]["stats"]["episodes"] > 0
