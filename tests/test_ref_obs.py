"""Reference-pose observations (EnvConfig.ref_obs_offsets, drl_set_ref_obs): one frame of reference qpos[1:] per offset
appended to every observation row.

Frame k of an observation built at cursor c is the reference qpos[1:] at the cursor reached by applying the cursor's
``next()`` k times to a copy of c, read with the episode's COM-Z shift: the target the pose reward compares against k
control steps later.  The float32 CPU reference below restates that over the oracle's RefCursor (and over
``LibraryRefCursor``, the per-clip cursor of a mocap library), literally: k calls of ``next()``.  The kernel advances
once per step transition instead; ``_advance_per_transition`` restates that loop and is held against the literal
definition.  A mirrored observation mirrors every frame with its own decision, through the qpos-block part of the
observation mirror table."""
import copy
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest

from drloco_b200 import lib
from drloco_b200.config import MOD_CUSTOM_POLICY, EnvConfig
from drloco_b200.ref_trajecs import loco3d_trajecs as l3
from drloco_b200.ref_trajecs import straight_walk_trajecs as sw
from drloco_b200.ref_trajecs.base_ref_trajecs import CURSOR_STEPWISE
from drloco_b200.walkers import MIRROR_OBS_IDX, make_spec, ref_frame_mirror_map
from oracle.env_oracle import RefCursor

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W3D, W165 = "StraightMimicWalker", "MimicWalker165cm65kg"


class LibraryRefCursor(RefCursor):
    """RefCursor over a library (the rules of tests/test_mocap_library.py): the walker3d wrap goes to the first step of
    the current clip, +1 after a right step; in wrap mode the cursor runs inside clip i_step."""

    def _clip_range(self, s):
        cf = self.t.clip_first_step
        k = int(np.searchsorted(cf, s, side="right")) - 1
        return int(cf[k]), int(cf[k + 1]) - 1

    def next(self):
        t = self.t
        if t.cursor_mode != CURSOR_STEPWISE:
            return super().next()
        self.pos += t.increment
        dif = self.pos - self.len + 1
        if dif > 0:
            first, last = self._clip_range(self.i_step)
            if self.i_step >= last:
                self.i_step = first + (0 if t.left_step[self.i_step] else 1)
            else:
                self.i_step += 1
                self.count_steps_same_vel += 1
            self.dist = float(t.step_last_comx[self.rsi_step])
            self.len = int(t.step_len[self.i_step])
            self.data_step = self.i_step
            self.pos = dif

    def init_random(self, i_step=None, pos=None):
        if self.t.cursor_mode == CURSOR_STEPWISE:
            return super().init_random(i_step, pos)
        self.i_step = int(i_step)
        self.len = int(self.t.step_len[self.i_step])
        self.pos = int(pos)
        self.data_step = self.shift_step = self.i_step
        self._begin_episode()


# --------------------------------------------------------------------------------------------------------------------
# the float32 CPU reference
# --------------------------------------------------------------------------------------------------------------------
def _qpos_f32(cur):
    """the kernel's reference qpos at the cursor: the float32 table row, COM-Z shifted in float32 (ref_lookup)"""
    t, nv = cur.t, cur.nv
    q = np.asarray(t.ref[int(t.step_off[cur.data_step]) + cur.pos, :nv], np.float32).copy()
    if t.cursor_mode != CURSOR_STEPWISE or cur.data_step == cur.shift_step:
        q[t.com_z_col] = np.float32(q[t.com_z_col] - np.float32(cur.z_off))
    return q


def ref_frames(cur, offsets, mirror_map=None):
    """[len(offsets), nv - 1] float32: frame k = qpos[1:] after k calls of next() on a copy of ``cur``; mirror_map =
    (idx, sign) of a mirrored observation"""
    c = copy.deepcopy(cur)
    out, done = [], 0
    for k in offsets:
        for _ in range(k - done):
            c.next()
        done = k
        f = _qpos_f32(c)[1:]
        if mirror_map is not None:
            idx, sgn = mirror_map
            f = (sgn * f[idx]).astype(np.float32)
        out.append(f)
    return np.stack(out)


def _advance_per_transition(cur, r):
    """the kernel's cursor advance (ref_obs_frames): r control steps in one iteration per step transition"""
    t, inc = cur.t, cur.t.increment
    while r > 0:
        ln = int(t.step_len[cur.data_step])
        room = ln - 1 - cur.pos
        if t.cursor_mode == CURSOR_STEPWISE:
            j = 1 if room < 0 else room // inc + 1
            if j > r:
                cur.pos += r * inc
                return
            if t.n_clips > 1:
                cf = t.clip_first_step
                k = int(np.searchsorted(cf, cur.i_step, side="right")) - 1
                first, last = int(cf[k]), int(cf[k + 1]) - 1
            else:
                first, last = 0, t.n_steps - 1
            cur.i_step = first + (0 if t.left_step[cur.i_step] else 1) if cur.i_step >= last else cur.i_step + 1
            cur.pos += j * inc - ln + 1
            cur.data_step = cur.i_step
            r -= j
        else:
            j = 1 if room <= 0 else -(-room // inc)
            if j > r:
                cur.pos += r * inc
                return
            cur.pos = 0
            r -= j


def _cursor(spec, i_step, pos, rsi_step=None, z_off=0.0, cls=RefCursor):
    c = cls(spec.mocap, spec.model.nv)
    c.init_random(rsi_step if rsi_step is not None else i_step, 0)
    c.i_step, c.pos = int(i_step), int(pos)
    c.data_step = int(i_step)
    c.len = int(spec.mocap.step_len[c.data_step])
    c.z_off = float(z_off)
    return c


def _clip_dir(tmp_path_factory):
    d = tmp_path_factory.mktemp("ref_obs_clips")
    for name, n, seed in (("s3.npz", 3, 11), ("s4.npz", 4, 12), ("s2.npz", 2, 13)):
        rows, lens = sw.synthetic_straight_rows(n_steps=n, seed=seed)
        np.savez(str(d / name), rows=rows, step_len=lens)
    return [str(d / "s3.npz"), str(d / "s4.npz"), str(d / "s2.npz")]


@pytest.fixture(scope="module")
def lib3(tmp_path_factory):
    return _clip_dir(tmp_path_factory)


@pytest.fixture(scope="module")
def lib165(tmp_path_factory):
    """a 2-clip loco3d (wrap-mode) library: i_step is the clip, the cursor wraps to 0 at the clip's own length"""
    d = tmp_path_factory.mktemp("ref_obs_loco3d")
    paths = []
    for name, seconds, seed in (("l6.npz", 6.0, 1), ("l9.npz", 9.0, 2)):
        ang, vel = l3.synthetic_loco3d(duration_s=seconds, seed=seed)
        np.savez(str(d / name), angJoi=ang, angDJoi=vel)
        paths.append(str(d / name))
    return paths


def _library_paths(library, lib3, lib165):
    return {False: None, "w3d": lib3, "w165": lib165}[library]


# --------------------------------------------------------------------------------------------------------------------
# CPU
# --------------------------------------------------------------------------------------------------------------------
def test_config_validation():
    assert EnvConfig().ref_obs_offsets == ()
    assert EnvConfig(ref_obs_offsets=[1, 5, 256]).ref_obs_offsets == (1, 5, 256)
    assert EnvConfig(ref_obs_offsets=(np.int64(3),)).ref_obs_offsets == (3,)
    for bad in ((0,), (257,), (-1,), (1.0,), (True,), ("1",), (2, 2), (5, 3), (1, 2, 3, 4), 5, "12", None):
        with pytest.raises(ValueError, match="ref_obs_offsets"):
            EnvConfig(ref_obs_offsets=bad)


def test_obs_dim_and_base_obs_dim():
    for env_id, base, nq in ((W3D, 29, 13), (W165, 47, 18)):
        for offs in ((), (1,), (1, 2), (4, 50, 256)):
            s = make_spec(EnvConfig(env_id=env_id, ref_obs_offsets=offs))
            assert s.base_obs_dim == base and s.obs_dim == base + len(offs) * nq
            assert len(s.mirror_tables()[0]) == base
    assert [29 + 13 * n for n in range(4)] == [29, 42, 55, 68]
    assert [47 + 18 * n for n in range(4)] == [47, 65, 83, 101]


def test_frame_mirror_map():
    s = make_spec(EnvConfig(env_id=W3D))
    idx, sgn = s.ref_frame_mirror()
    # columns 2..14 of the observation mirror table, relative to the block
    np.testing.assert_array_equal(idx, np.array(MIRROR_OBS_IDX[2:15]) - 2)
    np.testing.assert_array_equal(idx, [0, 1, 2, 3, 4, 9, 10, 11, 12, 5, 6, 7, 8])
    np.testing.assert_array_equal(np.nonzero(sgn < 0)[0] + 2, [2, 4, 6, 8, 12])
    assert sorted(idx.tolist()) == list(range(13))                  # a permutation of the block
    # mirroring off (and W165, which has none): the identity
    for cfg in (EnvConfig(env_id=W3D, modifications=(MOD_CUSTOM_POLICY,)), EnvConfig(env_id=W165)):
        idx, sgn = make_spec(cfg).ref_frame_mirror()
        assert (idx == np.arange(len(idx))).all() and (sgn == 1).all()
    bad = np.array(MIRROR_OBS_IDX)
    bad[5] = 16                                                     # reads a qvel column
    with pytest.raises(ValueError, match="qpos block"):
        ref_frame_mirror_map(bad, np.ones(29), 2, 13)
    bad[5] = 1                                                      # reads the desired velocity
    with pytest.raises(ValueError, match="qpos block"):
        ref_frame_mirror_map(bad, np.ones(29), 2, 13)


def test_per_transition_advance_equals_k_calls_of_next(lib3, lib165):
    """the kernel's loop against the literal definition, over random cursors of both walkers, a 3-clip walker3d
    library and a 2-clip loco3d library, including cursors past the end of their step and evaluation cursors reading
    step 0's table"""
    rng = np.random.default_rng(0)
    for spec, cls in ((make_spec(EnvConfig(env_id=W3D)), RefCursor), (make_spec(EnvConfig(env_id=W165)), RefCursor),
                      (make_spec(EnvConfig(env_id=W3D), lib3), LibraryRefCursor),
                      (make_spec(EnvConfig(env_id=W165), lib165), LibraryRefCursor)):
        t = spec.mocap
        for _ in range(400):
            s = int(rng.integers(0, t.n_steps))
            pos = int(rng.integers(0, t.step_len[s] + 3))
            c = _cursor(spec, s, pos, cls=cls)
            if t.cursor_mode == CURSOR_STEPWISE and rng.random() < 0.2:   # evaluation cursor: step 0's table
                c.data_step = c.shift_step = 0
                c.len = int(t.step_len[0])
            k = int(rng.integers(1, 257))
            a, b = copy.deepcopy(c), copy.deepcopy(c)
            for _ in range(k):
                a.next()
            _advance_per_transition(b, k)
            assert (a.i_step, a.pos, a.data_step) == (b.i_step, b.pos, b.data_step), (s, pos, k)


def test_cpu_reference_at_known_cursors(lib3):
    spec = make_spec(EnvConfig(env_id=W3D))
    t, inc = spec.mocap, spec.mocap.increment
    row = lambda s, p: np.asarray(t.ref[int(t.step_off[s]) + p, 1:14], np.float32)   # noqa: E731
    # mid-step: the rows k increments ahead in the same step; the COM-Z shift on the RSI step only
    c = _cursor(spec, 4, 100, rsi_step=4, z_off=0.25)
    f = ref_frames(c, (1, 3))
    want = row(4, 102).copy()
    want[1] = np.float32(want[1] - np.float32(0.25))
    np.testing.assert_array_equal(f[0], want)
    np.testing.assert_array_equal(f[1][[0, 2]], row(4, 106)[[0, 2]])
    c = _cursor(spec, 4, 100, rsi_step=3, z_off=0.25)                # another step's table is unshifted
    np.testing.assert_array_equal(ref_frames(c, (1,))[0], row(4, 102))
    # the last sample before a transition: pos = len - 1 - inc + 1 goes to the next step at pos dif
    ln = int(t.step_len[4])
    c = _cursor(spec, 4, ln - 2, rsi_step=0)
    np.testing.assert_array_equal(ref_frames(c, (1,))[0], row(5, 1))
    c = _cursor(spec, 4, ln - 3, rsi_step=0)
    np.testing.assert_array_equal(ref_frames(c, (1,))[0], row(4, ln - 1))
    # the last step wraps: +1 after a right step, to step 0 after a left one
    last = t.n_steps - 1
    ll = int(t.step_len[last])
    c = _cursor(spec, last, ll - 2, rsi_step=0)
    np.testing.assert_array_equal(ref_frames(c, (1,))[0], row(0 if t.left_step[last] else 1, 1))
    # a library clip's last step wraps inside the clip
    ls = make_spec(EnvConfig(env_id=W3D), lib3)
    lt = ls.mocap
    for k in range(lt.n_clips):
        s = int(lt.clip_first_step[k + 1]) - 1
        c = _cursor(ls, s, int(lt.step_len[s]) - 2, rsi_step=int(lt.clip_first_step[k]), cls=LibraryRefCursor)
        to = int(lt.clip_first_step[k]) + (0 if lt.left_step[s] else 1)
        np.testing.assert_array_equal(ref_frames(c, (1,))[0],
                                      np.asarray(lt.ref[int(lt.step_off[to]) + 1, 1:14], np.float32))
    # loco3d: pos wraps to 0, the COM-Z shift applies to the whole recording
    s165 = make_spec(EnvConfig(env_id=W165))
    t1, i1 = s165.mocap, s165.mocap.increment
    L1 = int(t1.step_len[0])
    c = _cursor(s165, 0, L1 - 1 - i1, z_off=0.125)
    f = ref_frames(c, (1, 2))
    w0 = np.asarray(t1.ref[0, :19], np.float32).copy()
    w0[2] = np.float32(w0[2] - np.float32(0.125))
    np.testing.assert_array_equal(f[0], w0[1:])
    w1 = np.asarray(t1.ref[i1, :19], np.float32).copy()
    w1[2] = np.float32(w1[2] - np.float32(0.125))
    np.testing.assert_array_equal(f[1], w1[1:])
    # evaluation mode: step 0's table and length until the first transition (the aliasing), then the logical step
    c = RefCursor(t, spec.model.nv)
    c.n_deterministic_inits = 5
    c.init_deterministic(20)
    c.adjust_COM_Z_pos(0.5)
    c.next()
    p0 = int(0.75 * int(t.step_len[5])) + inc
    np.testing.assert_array_equal(c.pos, p0)
    f = ref_frames(c, (1,))[0]
    want = row(0, p0 + inc).copy()
    want[1] = np.float32(want[1] - np.float32(0.5))                 # step 0's table got the shift
    np.testing.assert_array_equal(f, want)
    n_to = (int(t.step_len[0]) - 1 - p0) // inc + 1                 # calls of next() until the transition
    f = ref_frames(c, (n_to,))[0]
    np.testing.assert_array_equal(f, row(6, p0 + n_to * inc - int(t.step_len[0]) + 1))


def test_abi_argument_errors_without_a_device():
    if not os.path.exists(lib.LIB_PATH):
        import sys
        sys.path.insert(0, REPO)
        import __graft_entry__
        __graft_entry__.build()
    L = lib.load()
    offs = (C.c_int32 * 1)(1)
    assert L.drl_set_ref_obs(None, 1, C.cast(offs, C.c_void_p)) == -1          # DRL_ERR_INVALID
    assert b"null env" in L.drl_last_error()


# --------------------------------------------------------------------------------------------------------------------
# GPU
# --------------------------------------------------------------------------------------------------------------------
def _env(env_id, n, offs=(), paths=None, seed=5, **kw):
    from drloco_b200.vec_env import B200MimicVecEnv
    return B200MimicVecEnv(env_id, num_envs=n, cfg=EnvConfig(env_id=env_id, ref_obs_offsets=offs, **kw), seed=seed,
                           mocap_path=paths)


def _acts(n, act_dim, steps, seed):
    import torch
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.rand(steps, n, act_dim, device="cuda", generator=g) * 2 - 1


OFF_PATH_CASES = [
    (W3D, dict(integrator="rk4"), False),
    (W3D, dict(integrator="euler"), False),
    (W165, dict(integrator="rk4"), False),
    (W3D, dict(integrator="rk4", actuation="pd", pd_kp=200.0, pd_kv=5.0, contact_termination=True, ee_weight=0.15,
               adaptive_rsi=0.5), True),
]


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,kw,library", OFF_PATH_CASES, ids=["w3d-rk4", "w3d-euler", "w165-rk4", "w3d-lib3-all"])
def test_option_leaves_the_base_columns_alone(env_id, kw, library, lib3):
    """an env with 3 frames against one without, same seed and actions, 300 steps through B200VecNormalize: the base
    columns of obs and terminal_obs, reward, done, the normalised base columns and reward, stats, extras and state are
    bit-identical (VecNormalize statistics are per column)"""
    import torch
    from drloco_b200.vec_env import B200VecNormalize
    n, steps = 256, 300
    paths = lib3 if library else None
    runs = []
    for offs in ((), (1, 7, 40)):
        env = _env(env_id, n, offs, paths, seed=9, ep_dur_max=120, **kw)
        B = env.spec.base_obs_dim
        assert env.obs_dim == B + len(offs) * (env.spec.model.nv - 1)
        vn = B200VecNormalize(env)
        acts = _acts(n, env.act_dim, steps, 4)
        outs = [vn.reset_tensor()[:, :B].clone()]
        for a in acts:
            no, nr, d = vn.step_tensor(a)
            outs += [env.obs[:, :B].clone(), env.terminal_obs[:, :B].clone(), env.rew.clone(), d.float(),
                     no[:, :B].clone(), nr.clone()]
        q, v, c = env.get_state()
        om = vn.obs_rms
        runs.append(dict(outs=torch.cat([x.float().flatten() for x in outs]).cpu().numpy(), q=q, v=v, c=c,
                         stats=env.stats(), extras=env.extras().cpu().numpy(), mean=om.mean[:B], var=om.var[:B],
                         ret=(vn.ret_rms.mean, vn.ret_rms.var)))
        vn.close()
    a, b = runs
    for k in ("outs", "q", "v", "c", "extras", "mean", "var"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert a["stats"] == b["stats"] and a["ret"] == b["ret"]
    assert a["stats"]["episodes"] > 0


def _frames_of(rows, spec):
    nq = spec.model.nv - 1
    return rows[:, spec.base_obs_dim:].reshape(len(rows), -1, nq)


FRAME_CASES = [
    (W3D, (1,), {}, False), (W3D, (3, 40, 256), {}, False),
    (W3D, (2, 17, 100), dict(modifications=(MOD_CUSTOM_POLICY,)), False),
    (W165, (1,), {}, False), (W165, (5, 60, 256), {}, False),
    (W3D, (1,), {}, "w3d"), (W3D, (7, 90, 200), {}, "w3d"),
    (W165, (1,), {}, "w165"), (W165, (5, 60, 256), {}, "w165"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,offs,kw,library", FRAME_CASES,
                         ids=["w3d-1", "w3d-3", "w3d-nomirror-3", "w165-1", "w165-3", "lib3-1", "lib3-3", "lib165-1",
                              "lib165-3"])
def test_frames_equal_the_cpu_reference(env_id, offs, kw, library, lib3, lib165):
    """logic-only steps (frame_skip 0) from injected cursors, edge cursors included (the last samples of a step, the
    last step of every clip, the loco3d wrap): every frame column of obs and terminal_obs equals the float32 CPU
    reference exactly, mirrored with the observation's own decision"""
    n, rounds, ep_max = 96, 6, 1000
    env = _env(env_id, n, offs, _library_paths(library, lib3, lib165), ep_dur_max=ep_max, **kw)
    env.debug_set(frame_skip_override=0)
    spec, t = env.spec, env.spec.mocap
    cls = LibraryRefCursor if library else RefCursor
    mm = spec.ref_frame_mirror()
    mirror = spec.mirror

    def want(cur):
        left = mirror and bool(t.left_step[cur.i_step])
        return ref_frames(cur, offs, mm if left else None)

    rng = np.random.default_rng(3)
    istep = rng.integers(0, t.n_steps, n).astype(np.int32)
    pos = np.array([rng.integers(0, t.step_len[i]) for i in istep], np.int32)
    obs = env.reset(inject=(istep, pos))
    zoff = env.extras().cpu().numpy()[:, 7]
    cur = []
    for i in range(n):
        c = cls(t, spec.model.nv)
        c.init_random(int(istep[i]), int(pos[i]))
        c.adjust_COM_Z_pos(float(zoff[i]))
        c.next()
        cur.append(c)
    got = env.get_state()[2]
    assert all((got[i, 0], got[i, 1]) == (cur[i].i_step, cur[i].pos) for i in range(n))
    fr = _frames_of(obs.astype(np.float32), spec)
    for i in range(n):
        np.testing.assert_array_equal(fr[i], want(cur[i]), err_msg=f"reset, env {i}")
    inc = t.increment
    zero = np.zeros((n, env.act_dim), np.float32)
    n_term = 0
    for r in range(rounds):
        # edge cursors: a step's last samples (a transition within the first frame), every clip's last step
        cset = env.get_state()[2].copy()
        for i in range(n):
            s = int(rng.integers(0, t.n_steps))
            if t.cursor_mode != CURSOR_STEPWISE:
                s = cur[i].i_step                   # loco3d: the clip of the episode, wrapping at its own length
            elif i < t.n_clips:
                s = int(t.clip_first_step[i + 1]) - 1
            ln = int(t.step_len[s])
            choice = [ln // 2, ln - 1 - 2 * inc, ln - 1 - inc, ln - 2, 0, int(rng.integers(0, ln))]
            p = choice[(i + r) % len(choice)]
            cset[i, 0], cset[i, 1] = s, p
            cset[i, 3] = ep_max - 1 if (i + r) % 3 == 0 else 5      # a third of the envs time out on this step
        env.set_state(cursor=cset)
        for i in range(n):
            c = cur[i]
            c.i_step, c.pos = int(cset[i, 0]), int(cset[i, 1])
            c.data_step = c.i_step
            c.len = int(t.step_len[c.i_step])
            c.next()
        o, _, d, infos = env.step(zero, inject=(istep, pos))
        o = o.astype(np.float32)
        to = np.zeros_like(o)
        for i in np.nonzero(d)[0]:
            to[i] = infos[i]["terminal_observation"]
        assert d.sum() == sum((i + r) % 3 == 0 for i in range(n))
        zoff = env.extras().cpu().numpy()[:, 7]
        fo, ft = _frames_of(o, spec), _frames_of(to, spec)
        for i in range(n):
            if d[i]:
                np.testing.assert_array_equal(ft[i], want(cur[i]), err_msg=f"terminal, round {r}, env {i}")
                c = cls(t, spec.model.nv)
                c.init_random(int(istep[i]), int(pos[i]))
                c.adjust_COM_Z_pos(float(zoff[i]))
                c.next()
                cur[i] = c
                n_term += 1
            np.testing.assert_array_equal(fo[i], want(cur[i]), err_msg=f"obs, round {r}, env {i}, done {d[i]}")
        got = env.get_state()[2]
        assert all((got[i, 0], got[i, 1]) == (cur[i].i_step, cur[i].pos) for i in range(n))
    assert n_term > 0
    env.close()


@pytest.mark.gpu
def test_frames_in_evaluation_mode_follow_the_step0_aliasing():
    """deterministic inits read step 0's table (and its COM-Z shift) until the first transition; the frames of the
    reset and of the following logic-only steps equal the CPU reference's k calls of next()"""
    offs = (1, 30, 256)
    n = 20
    env = _env(W3D, n, offs)
    env.debug_set(frame_skip_override=0)
    spec, t = env.spec, env.spec.mocap
    mm = spec.ref_frame_mirror()
    env.env_method("activate_evaluation")
    env.set_det_init_counters(np.arange(n) % env.cfg.eval_n_times)
    obs = env.reset()
    zoff = env.extras().cpu().numpy()[:, 7]
    cur = []
    for i in range(n):
        c = RefCursor(t, spec.model.nv)
        c.n_deterministic_inits = i % env.cfg.eval_n_times
        c.init_deterministic(env.cfg.eval_n_times)
        c.adjust_COM_Z_pos(float(zoff[i]))
        c.next()
        cur.append(c)
    zero = np.zeros((n, env.act_dim), np.float32)
    for k in range(120):
        fr = _frames_of(obs.astype(np.float32), spec)
        for i in range(n):
            left = bool(t.left_step[cur[i].i_step])
            np.testing.assert_array_equal(fr[i], ref_frames(cur[i], offs, mm if left else None), err_msg=f"{k} {i}")
        obs, _, done, _ = env.step(zero)
        assert not done.any()
        for c in cur:
            c.next()
    assert all(c.data_step == c.i_step for c in cur)           # every env has passed its first transition
    env.close()


def _unmirror(block, idx, sgn):
    x = np.empty_like(block)
    x[..., idx] = sgn * block
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,library", [(W3D, False), (W165, False), (W3D, "w3d"), (W165, "w165")],
                         ids=["w3d", "w165", "lib3", "lib165"])
def test_playback_frames_are_the_future_qpos(env_id, library, lib3, lib165):
    """playback: frame k at step t, un-mirrored with the step's own flag, equals bit for bit the un-mirrored qpos
    block of the observation at step t + k for every env whose episode does not end in (t, t + k]"""
    offs = (1, 4, 16)
    n, steps = 128, 260
    env = _env(env_id, n, offs, _library_paths(library, lib3, lib165), seed=2, ep_dur_max=150)
    spec, t = env.spec, env.spec.mocap
    idx, sgn = spec.ref_frame_mirror()
    Bq, nq = spec.qpos_block, spec.model.nv - 1
    env.set_playback(True)
    O, L, D = [], [], []
    obs = env.reset()
    dn = np.zeros(n, bool)
    zero = np.zeros((n, env.act_dim), np.float32)
    for _ in range(steps):
        cur = env.get_state()[2]
        O.append(obs.astype(np.float32))
        L.append(spec.mirror & t.left_step[cur[:, 0]].astype(bool))
        D.append(dn)
        obs, _, dn, _ = env.step(zero)
    O, L, D = np.stack(O), np.stack(L), np.stack(D)
    un = lambda x, left: np.where(left[:, None], _unmirror(x, idx, sgn), x)   # noqa: E731
    checked = 0
    for ti in range(steps):
        fr = _frames_of(O[ti], spec)
        for f, k in enumerate(offs):
            if ti + k >= steps:
                continue
            ok = ~D[ti + 1:ti + k + 1].any(axis=0)
            a = un(fr[:, f], L[ti])
            b = un(O[ti + k][:, Bq:Bq + nq], L[ti + k])
            np.testing.assert_array_equal(a[ok], b[ok], err_msg=f"step {ti}, offset {k}")
            checked += int(ok.sum())
    assert checked > n * steps
    assert D.any()
    env.set_playback(False)
    env.close()


def _reductions_module():
    spec = importlib.util.spec_from_file_location("_reductions_at_scale",
                                                  os.path.join(REPO, "tests", "test_reductions_at_scale.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("walker,n", [(W3D, 4096), (W3D, 65536), (W165, 4096)])
def test_full_width_moments_against_float64(walker, n):
    """the step kernel's fused moments over the whole row (base and frame columns): the VecNormalize statistics
    against a float64 RunningMeanStd of the raw observations, to the bound of tests/test_reductions_at_scale.py"""
    import torch
    from drloco_b200.vec_env import B200VecNormalize
    from oracle.env_oracle import RunningMeanStd
    R = _reductions_module()
    env = _env(walker, n, (1, 9, 50), seed=7, ep_dur_max=40)
    _, epb, _, _, ngroups, _ = R._launch_shape(walker, n, 128)
    depth = R._epilogue_depth(epb, ngroups)
    vn = B200VecNormalize(env)
    D = env.obs_dim
    obs_rms = RunningMeanStd(shape=(D,))
    ob = R._RmsBound(depth, (D,))
    vn.reset_tensor()
    rng = np.random.default_rng(n)
    n_done = 0
    for k in range(50):
        act = torch.as_tensor(rng.uniform(-1, 1, (n, env.act_dim)).astype(np.float32), device=env.device)
        _, _, done = vn.step_tensor(act)
        raw = env.obs.cpu().numpy()
        n_done += int(done.sum())
        obs_rms.update(raw.astype(np.float64))
        ob.add(raw)
        om = vn.obs_rms
        assert om.count == obs_rms.count
        ob.check(om.mean, om.var, obs_rms, f"obs_rms, step {k}")
    assert n_done > 0
    vn.close()


@pytest.mark.gpu
def test_determinism_and_graph_path(lib3):
    """two runs bit-identical; the CUDA-graph numpy path of B200VecNormalize equals its eager tensor path"""
    import torch
    from drloco_b200.vec_env import vec_env
    n, steps = 512, 80
    cfg = EnvConfig(env_id=W3D, ref_obs_offsets=(2, 20, 200), ep_dur_max=60)
    rng = np.random.default_rng(5)
    acts = rng.uniform(-1, 1, (steps, n, 8)).astype(np.float32)
    runs = []
    for mode in ("graph", "graph", "tensor"):
        v = vec_env(W3D, num_envs=n, seed=8, mocap_path=lib3, cfg=cfg)
        outs = []
        if mode == "graph":
            assert v.use_graph
            outs.append(v.reset())
            for a in acts:
                o, r, d, infos = v.step(a)
                term = np.zeros((n, v.venv.obs_dim), np.float32)
                for i in np.nonzero(d)[0]:
                    term[i] = infos[i]["terminal_observation"]
                outs += [o, r, d, term]
            assert v.use_graph
        else:
            outs.append(v.reset_tensor().cpu().numpy())
            for a in acts:
                o, r, d = v.step_tensor(torch.as_tensor(a, device="cuda"))
                dd = d.cpu().numpy().astype(bool)
                rms = v._rms[v._cur].cpu().numpy()
                D = v._D
                to = v.venv.terminal_obs.cpu().numpy()
                inv = (1.0 / np.sqrt(rms[D:2 * D] + np.float32(v.epsilon))).astype(np.float32)
                tn = np.clip((to - rms[:D].astype(np.float32)) * inv, -v.clip_obs, v.clip_obs).astype(np.float32)
                outs += [o.cpu().numpy(), r.cpu().numpy(), dd, np.where(dd[:, None], tn, 0).astype(np.float32)]
        runs.append([np.asarray(x, np.float64) for x in outs])
        v.close()
    for a, b in zip(runs[0], runs[1]):
        np.testing.assert_array_equal(a, b)
    for j, (a, b) in enumerate(zip(runs[0], runs[2])):
        if j % 4 == 0 and j > 0:          # terminal observations: the host restatement of the normalisation
            np.testing.assert_allclose(a, b, rtol=1e-6, atol=1e-6)
        else:
            np.testing.assert_array_equal(a, b)
    assert sum(x.sum() for x in runs[0][3::4]) > 0


@pytest.mark.gpu
def test_abi_call_order_and_argument_errors():
    import torch
    from drloco_b200 import cabi
    from drloco_b200.vec_env import B200VecNormalize
    L = lib.load()
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    one = np.array([1], np.int32)
    env = _env(W3D, 8)
    # before drl_upload_model: a raw env of the same configuration
    h = C.c_void_p()
    c = env._make_config(5, 0, 0)
    lib.check(L.drl_create(C.byref(c), C.byref(h)), "drl_create")
    assert L.drl_set_ref_obs(h, 1, p(one)) == -3
    lib.check(L.drl_upload_model(h, C.byref(cabi.pack_model(env.spec.model))), "drl_upload_model")
    for n, offs in ((1, [0]), (1, [257]), (2, [3, 3]), (2, [5, 2]), (4, [1, 2, 3, 4]), (-1, [1])):
        assert L.drl_set_ref_obs(h, n, p(np.array(offs, np.int32))) == -1, offs
    assert L.drl_set_ref_obs(h, 1, None) == -1
    lib.check(L.drl_set_ref_obs(h, 3, p(np.array([1, 2, 256], np.int32))), "drl_set_ref_obs")
    lib.check(L.drl_set_ref_obs(h, 0, None), "drl_set_ref_obs")
    L.drl_destroy(h)
    # a mirror table that leaves the qpos block
    c = env._make_config(5, 0, 0)
    c.mirror_obs_idx[7] = 20
    h = C.c_void_p()
    lib.check(L.drl_create(C.byref(c), C.byref(h)), "drl_create")
    lib.check(L.drl_upload_model(h, C.byref(cabi.pack_model(env.spec.model))), "drl_upload_model")
    assert L.drl_set_ref_obs(h, 1, p(one)) == -1
    assert b"qpos block" in L.drl_last_error()
    L.drl_destroy(h)
    # after the first reset; while a VecNormalize is attached
    env.reset()
    assert L.drl_set_ref_obs(env._handle, 1, p(one)) == -3
    env.close()
    env = _env(W3D, 8)
    vn = B200VecNormalize(env)
    assert L.drl_set_ref_obs(env._handle, 1, p(one)) == -3
    # a failed call changed nothing: the rows keep the base width
    o = vn.reset_tensor()
    assert o.shape == (8, 29)
    o, _, _ = vn.step_tensor(torch.zeros(8, env.act_dim, device="cuda"))
    assert torch.isfinite(o).all()
    vn.close()


@pytest.mark.gpu
def test_loading_statistics_of_another_width_raises(tmp_path):
    from drloco_b200.vec_env import B200VecNormalize
    v29 = B200VecNormalize(_env(W3D, 8))
    path = str(tmp_path / "vn29.pkl")
    v29.save(path)
    sd = v29.state_dict()
    v29.close()
    env42 = _env(W3D, 8, (5,))
    with pytest.raises(ValueError, match=r"29.*42"):
        B200VecNormalize.load(path, env42)
    # the refused file left the env unattached: the setter, refused while a VecNormalize is attached, still accepts
    # the env's own configuration, and a wrapper of the right width then steps it
    offs = np.array([5], np.int32)
    lib.check(lib.load().drl_set_ref_obs(env42._handle, 1, offs.ctypes.data_as(C.c_void_p)), "drl_set_ref_obs")
    v = B200VecNormalize(env42)
    import torch
    v.reset_tensor()
    o, _, _ = v.step_tensor(torch.zeros(8, env42.act_dim, device="cuda"))
    assert o.shape == (8, 42) and bool(torch.isfinite(o).all())
    v.close()
    v42 = B200VecNormalize(_env(W3D, 8, (5,)))
    with pytest.raises(ValueError, match=r"29.*42"):
        v42.load_state_dict(sd)
    v42.close()
