"""Mocap libraries: several recordings of one walker in one batch (make_spec(mocap_path=[...]), drl_set_mocap_clips).

A library is an ordered list of clips, each compiled from one file as before.  An episode stays in the clip it started
in: the walker3d wrap (straight_walk_trajecs.py:330-333) and the desired-velocity clamp act per clip, and in the loco3d
(wrap) mode every clip is one step whose desired-velocity window never crosses into the next clip.  RSI draws a clip
with probability proportional to its weight (default: its sample count), then the reference's draw inside it.  With
one clip every output is the single recording's, bit for bit.

No second real recording ships with the repository: the clips below are the shipped constant-speed file, synthetic
straight-walking gaits saved as .npz and as the reference's 40-row ramp .mat layout, and synthetic loco3d recordings of
different lengths and seeds.  `LibraryRefCursor` restates the per-clip cursor rules on top of the oracle's RefCursor;
the GPU cursor is held against it."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest
import scipy.io as spio
from scipy import stats as sps

from drloco_b200 import lib
from drloco_b200.config import EnvConfig
from drloco_b200.ref_trajecs import loco3d_trajecs as l3
from drloco_b200.ref_trajecs import straight_walk_trajecs as sw
from drloco_b200.ref_trajecs.base_ref_trajecs import CURSOR_STEPWISE, clip_weights, concat_tables
from drloco_b200.vec_env import ADAPTIVE_RSI_BIN_STEPS, adaptive_rsi_bins
from drloco_b200.walkers import make_spec
from oracle.env_oracle import RefCursor

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W3D, W165 = "StraightMimicWalker", "MimicWalker165cm65kg"
ALPHA = 1e-3        # significance level of the chi-square tests (fixed seeds: the outcome is deterministic)


# --------------------------------------------------------------------------------------------------------------------
# clip files
# --------------------------------------------------------------------------------------------------------------------
def _straight_npz(path, n_steps, seed):
    rows, lens = sw.synthetic_straight_rows(n_steps=n_steps, seed=seed)
    np.savez(path, rows=rows, step_len=lens)
    return rows, lens


def _ramp_mat(path, n_steps, seed):
    """the synthetic 38-row gait re-laid out as the reference's 40-row ramp file: two GRF rows inserted at 35-36"""
    rows38, lens = sw.synthetic_straight_rows(n_steps=n_steps, seed=seed)
    off = np.concatenate([[0], np.cumsum(lens)])
    data = np.empty(n_steps, dtype=object)
    for i in range(n_steps):
        s = rows38[:, off[i]:off[i + 1]]
        grf = np.stack([700.0 + 50.0 * np.sin(np.linspace(0, np.pi, s.shape[1])), np.zeros(s.shape[1])])
        data[i] = np.concatenate([s[:35], grf, s[35:38]], axis=0)
    spio.savemat(path, {"Data": data})
    return rows38, lens


def _loco3d_npz(path, seconds, seed):
    ang, vel = l3.synthetic_loco3d(duration_s=seconds, seed=seed)
    np.savez(path, angJoi=ang, angDJoi=vel)
    return ang, vel


@pytest.fixture(scope="module")
def clip_dir(tmp_path_factory):
    d = tmp_path_factory.mktemp("clips")
    _straight_npz(str(d / "s3.npz"), 3, 11)
    _ramp_mat(str(d / "ramp4.mat"), 4, 12)
    _straight_npz(str(d / "s2.npz"), 2, 13)
    _loco3d_npz(str(d / "l6.npz"), 6.0, 1)
    _loco3d_npz(str(d / "l9.npz"), 9.0, 2)
    return d


def _w3d_paths(d):
    return [str(d / "s3.npz"), str(d / "ramp4.mat"), str(d / "s2.npz")]


def _w165_paths(d):
    return [str(d / "l6.npz"), str(d / "l9.npz")]


# --------------------------------------------------------------------------------------------------------------------
# the per-clip cursor, restated over the oracle's RefCursor
# --------------------------------------------------------------------------------------------------------------------
class LibraryRefCursor(RefCursor):
    """RefCursor over a library: the walker3d wrap goes to the first step (+1 for a right step) of the current clip,
    the desired-velocity step is clamped at the clip's first step, and in wrap mode the cursor runs inside clip
    i_step, whose desired-velocity window is the clip's slice of the rows; an injected istep picks the clip there."""

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

    def get_desired_walking_velocity_vector(self):
        t = self.t
        if t.cursor_mode == CURSOR_STEPWISE:
            first, _ = self._clip_range(self.i_step)
            return [float(t.step_vel[max(first, self.i_step - self.count_steps_same_vel + 1)])]
        end = min(self.pos + t.des_vel_window, self.len - 1)
        n = end - self.pos
        if n <= 0:
            return [math.nan, math.nan]
        off = int(t.step_off[self.i_step])
        rows = t.des_vel_rows
        return [np.mean(rows[0, off + self.pos:off + end]), np.mean(rows[1, off + self.pos:off + end])]

    def init_random(self, i_step=None, pos=None):
        if self.t.cursor_mode == CURSOR_STEPWISE:
            return super().init_random(i_step, pos)
        self.i_step = int(i_step)
        self.len = int(self.t.step_len[self.i_step])
        self.pos = int(pos)
        self.data_step = self.shift_step = self.i_step
        self._begin_episode()


def _host_des_vel(t, i_step, pos):
    """the kernel's loco3d desired velocity from the library's prefix sums (float64 difference / n, then float32)"""
    ln = int(t.step_len[i_step])
    end = min(pos + t.des_vel_window, ln - 1)
    n = end - pos
    if n <= 0:
        return np.float32(np.nan)
    base = int(t.step_off[i_step]) + i_step
    pre = t.des_vel_prefix
    return np.float32((pre[base + end, 0] - pre[base + pos, 0]) / float(n))


# --------------------------------------------------------------------------------------------------------------------
# CPU: tables
# --------------------------------------------------------------------------------------------------------------------
def test_concat_tables_offsets_and_lengths(clip_dir):
    cfg = EnvConfig(env_id=W3D)
    paths = _w3d_paths(clip_dir)
    parts = [make_spec(cfg, p).mocap for p in paths]
    lib_t = make_spec(cfg, paths).mocap
    assert lib_t.n_clips == 3 and [t.n_clips for t in parts] == [1, 1, 1]
    np.testing.assert_array_equal(lib_t.clip_first_step, [0, 3, 7, 9])
    assert lib_t.n_steps == 9 and lib_t.n_samples == sum(t.n_samples for t in parts)
    s0 = 0
    for k, t in enumerate(parts):
        a = lib_t.clip_first_step[k]
        np.testing.assert_array_equal(lib_t.step_off[a:a + t.n_steps], t.step_off + s0)
        for name in ("step_len", "left_step", "step_vel", "step_last_comx"):
            np.testing.assert_array_equal(getattr(lib_t, name)[a:a + t.n_steps], getattr(t, name), err_msg=name)
        np.testing.assert_array_equal(lib_t.ref[s0:s0 + t.n_samples], t.ref)
        s0 += t.n_samples
    # default weights: proportional to the sample counts
    ns = np.array([t.n_samples for t in parts], np.float64)
    np.testing.assert_allclose(lib_t.clip_weight, ns / ns.sum(), rtol=1e-15)
    np.testing.assert_allclose(make_spec(cfg, paths, [1, 0, 3]).mocap.clip_weight, [0.25, 0, 0.75], rtol=1e-15)


def test_single_path_list_is_the_single_recording(clip_dir):
    for env_id, p in ((W3D, None), (W3D, str(clip_dir / "ramp4.mat")), (W165, str(clip_dir / "l6.npz"))):
        a = make_spec(EnvConfig(env_id=env_id), p).mocap
        b = make_spec(EnvConfig(env_id=env_id), [p]).mocap
        assert a.n_clips == b.n_clips == 1
        for name in ("ref", "step_off", "step_len", "left_step", "step_vel", "step_last_comx", "des_vel_prefix",
                     "des_vel_rows", "clip_first_step", "clip_weight"):
            x, y = getattr(a, name), getattr(b, name)
            assert (x is None and y is None) or np.array_equal(x, y), name


def test_loco3d_prefix_sums_restart_per_clip(clip_dir):
    paths = _w165_paths(clip_dir)
    cfg = EnvConfig(env_id=W165)
    parts = [make_spec(cfg, p).mocap for p in paths]
    t = make_spec(cfg, paths).mocap
    np.testing.assert_array_equal(t.clip_first_step, [0, 1, 2])
    np.testing.assert_array_equal(t.step_off, [0, parts[0].n_samples])
    assert t.des_vel_prefix.shape == (t.n_samples + 2, 2)
    base1 = parts[0].n_samples + 1
    np.testing.assert_array_equal(t.des_vel_prefix[0], [0, 0])
    np.testing.assert_array_equal(t.des_vel_prefix[base1], [0, 0])
    np.testing.assert_array_equal(t.des_vel_prefix[base1:], parts[1].des_vel_prefix)
    # a window near the end of clip 0 is the mean of clip 0's slice only, never of clip 1's first samples
    vel0 = np.load(paths[0])["angDJoi"]
    ln0 = int(t.step_len[0])
    for pos in (ln0 - 300, ln0 - 100, ln0 - 2):
        end = min(pos + t.des_vel_window, ln0 - 1)
        want = np.mean(vel0[l3.PELVIS_TX, pos:end])
        got = (t.des_vel_prefix[end, 0] - t.des_vel_prefix[pos, 0]) / (end - pos)
        assert np.isclose(got, want, rtol=1e-10, atol=1e-13)
        c = LibraryRefCursor(t, 19)
        c.init_random(0, pos)
        assert c.get_desired_walking_velocity_vector()[0] == want
    # the same in clip 1, through the cursor restatement (row offset of clip 1)
    vel1 = np.load(paths[1])["angDJoi"]
    c = LibraryRefCursor(t, 19)
    c.init_random(1, int(t.step_len[1]) - 50)
    assert c.get_desired_walking_velocity_vector()[0] == np.mean(vel1[l3.PELVIS_TX, int(t.step_len[1]) - 50:-1])
    c.init_random(1, int(t.step_len[1]) - 1)
    assert math.isnan(c.get_desired_walking_velocity_vector()[0])           # Q23 per clip


def test_38_and_40_row_clips_of_the_same_motion_give_identical_rows(tmp_path):
    npz, mat = str(tmp_path / "a.npz"), str(tmp_path / "a.mat")
    _straight_npz(npz, 5, 21)
    _ramp_mat(mat, 5, 21)
    t = make_spec(EnvConfig(env_id=W3D), [npz, mat]).mocap
    n = t.n_samples // 2
    np.testing.assert_array_equal(t.ref[:n], t.ref[n:])
    for name in ("step_len", "left_step", "step_vel", "step_last_comx"):
        x = getattr(t, name)
        np.testing.assert_array_equal(x[:5], x[5:], err_msg=name)


def test_concat_tables_rejects_mixed_libraries(clip_dir):
    w3d = make_spec(EnvConfig(env_id=W3D), str(clip_dir / "s3.npz")).mocap
    w165 = make_spec(EnvConfig(env_id=W165), str(clip_dir / "l6.npz")).mocap
    with pytest.raises(ValueError):
        concat_tables([])
    with pytest.raises(ValueError, match="cursor_mode"):
        concat_tables([w3d, w165])
    import dataclasses
    for name, val in (("increment", 4), ("com_z_col", 1)):
        with pytest.raises(ValueError, match=name):
            concat_tables([w3d, dataclasses.replace(w3d, **{name: val})])
    with pytest.raises(ValueError, match="des_vel_window"):
        concat_tables([w165, dataclasses.replace(w165, des_vel_window=10)])
    one_step = dataclasses.replace(w3d, step_off=w3d.step_off[:1], step_len=w3d.step_len[:1],
                                   left_step=w3d.left_step[:1], step_vel=w3d.step_vel[:1],
                                   step_last_comx=w3d.step_last_comx[:1], clip_first_step=None)
    with pytest.raises(ValueError, match="at least 2"):
        concat_tables([w3d, one_step])
    with pytest.raises(ValueError, match="already a library"):
        concat_tables([concat_tables([w3d, w3d]), w3d])


def test_clip_weight_validation(clip_dir):
    paths = _w3d_paths(clip_dir)
    for bad in ([1, 2], [1, -1, 1], [0, 0, 0], [1, float("nan"), 1], [1, float("inf"), 1]):
        with pytest.raises(ValueError):
            make_spec(EnvConfig(env_id=W3D), paths, bad)
    with pytest.raises(ValueError):
        make_spec(EnvConfig(env_id=W3D), None, [-1.0])                   # one clip: validated, then always drawn
    with pytest.raises(ValueError):
        make_spec(EnvConfig(env_id=W3D), [])
    np.testing.assert_array_equal(clip_weights(None, [10, 30]), [0.25, 0.75])


def test_adaptive_rsi_bins_over_a_library(clip_dir):
    """u_b = w_c / steps_c * width_b / step length: sums to 1, and equals a float64 model of the base draw"""
    t = make_spec(EnvConfig(env_id=W3D), _w3d_paths(clip_dir), [0.5, 0.2, 0.3]).mocap
    bs = ADAPTIVE_RSI_BIN_STEPS * t.increment
    b = adaptive_rsi_bins(t.step_len, bs, t.clip_first_step, t.clip_weight)
    assert np.isclose(b["u"].sum(), 1.0, rtol=0, atol=1e-12)
    cf = t.clip_first_step
    for k, w in enumerate([0.5, 0.2, 0.3]):
        steps = np.arange(cf[k], cf[k + 1])
        assert np.isclose(b["u"][np.isin(b["step"], steps)].sum(), w, rtol=1e-12)
    # model: probability of every sample under the base draw, summed over the bin
    for i in range(len(b["u"])):
        s = int(b["step"][i])
        k = int(np.searchsorted(cf, s, side="right")) - 1
        p = t.clip_weight[k] / (cf[k + 1] - cf[k]) / t.step_len[s]
        assert np.isclose(b["u"][i], p * b["width"][i], rtol=1e-14)
    # one clip: the single-recording table, bit for bit
    t1 = make_spec(EnvConfig(env_id=W3D)).mocap
    a1 = adaptive_rsi_bins(t1.step_len, bs)
    b1 = adaptive_rsi_bins(t1.step_len, bs, t1.clip_first_step, t1.clip_weight)
    np.testing.assert_array_equal(a1["u"], b1["u"])


@pytest.fixture(scope="module")
def built_lib():
    if not os.path.exists(lib.LIB_PATH):
        sys.path.insert(0, REPO)
        import __graft_entry__
        __graft_entry__.build()
    return lib.load()


def test_abi_argument_errors_without_a_device(built_lib):
    L = built_lib
    first = (C.c_int32 * 3)(0, 2, 4)
    w = (C.c_double * 2)(1.0, 1.0)
    assert L.drl_set_mocap_clips(None, 2, C.cast(first, C.c_void_p), C.cast(w, C.c_void_p)) == -1   # DRL_ERR_INVALID
    assert b"null argument" in L.drl_last_error()
    out = (C.c_int64 * 10)()
    assert L.drl_get_clip_stats(None, C.cast(out, C.c_void_p), None) == -1
    assert b"null argument" in L.drl_last_error()


# --------------------------------------------------------------------------------------------------------------------
# GPU
# --------------------------------------------------------------------------------------------------------------------
def _gpu_env(env_id, n, paths=None, weights=None, seed=5, **kw):
    from drloco_b200.vec_env import B200MimicVecEnv
    return B200MimicVecEnv(env_id, num_envs=n, cfg=EnvConfig(env_id=env_id, **kw), seed=seed, mocap_path=paths,
                           clip_weights=weights)


def _acts(n, act_dim, steps, seed):
    import torch
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.rand(steps, n, act_dim, device="cuda", generator=g) * 2 - 1


def _run_tensor(env, acts):
    import torch
    outs = [env.reset_tensor().clone()]
    for a in acts:
        o, r, d = env.step_tensor(a)
        outs += [o.clone(), r.clone(), d.clone(), env.terminal_obs.clone()]
    q, v, c = env.get_state()
    rec = env.episode_records()
    return dict(outs=torch.cat([x.float().flatten() for x in outs]).cpu().numpy(), q=q, v=v, c=c, stats=env.stats(),
                extras=env.extras().cpu().numpy(), ring=sorted(zip(*(rec[k].tolist() for k in sorted(rec)))))


def _clip_of(t, steps):
    return np.searchsorted(t.clip_first_step, steps, side="right") - 1


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,kw", [
    (W3D, dict(integrator="rk4")), (W3D, dict(integrator="euler")), (W165, dict(integrator="rk4")),
    (W3D, dict(integrator="rk4", actuation="pd", pd_kp=200.0, pd_kv=5.0, contact_termination=True, ee_weight=0.15,
               adaptive_rsi=0.5))])
def test_single_clip_list_is_the_single_recording_on_the_gpu(env_id, kw):
    """mocap_path=[p] against mocap_path=p: obs, reward, done, terminal obs, state, statistics, extras and the episode
    ring, bit for bit over 200 random-action steps"""
    n, steps = 256, 200
    acts = _acts(n, make_spec(EnvConfig(env_id=env_id, **kw)).act_dim, steps, 4)
    runs = []
    for paths in (None, [None]):
        env = _gpu_env(env_id, n, paths, seed=9, **kw)
        runs.append(_run_tensor(env, acts))
        env.close()
    a, b = runs
    for k in ("outs", "q", "v", "c", "extras"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert a["stats"] == b["stats"] and a["ring"] == b["ring"]


def _library_oracle(spec, n):
    from oracle.env_oracle import OracleVecEnv
    from oracle.physics import OraclePhysics

    class Frozen:
        def __init__(self):
            self._p = OraclePhysics(spec.model)
            self.qacc_warm = self._p.qacc_warm

        def step(self, q, v, ctrl, nsub):
            return False

        def site_xpos(self, q):
            return self._p.site_xpos(q)

    ora = OracleVecEnv(spec, n, Frozen)
    for e in ora.envs:
        e.env.refs = LibraryRefCursor(spec.mocap, spec.model.nv)
    return ora


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", [W3D, W165])
def test_cursor_parity_with_the_oracle(clip_dir, env_id):
    """logic-only steps (frame_skip 0) over a 3-clip walker3d / 2-clip loco3d library with injected draws, long enough
    for every clip to wrap: cursor, phase, desired velocity, mirroring and done bit-exact against LibraryRefCursor,
    observations within the logic tests' tolerance"""
    paths = _w3d_paths(clip_dir) if env_id == W3D else _w165_paths(clip_dir)
    n, steps = 12, 2000
    ep_max = 700 if env_id == W3D else 1300
    env = _gpu_env(env_id, n, paths, ep_dur_max=ep_max)
    t = env.spec.mocap
    env.debug_set(frame_skip_override=0)
    ora = _library_oracle(env.spec, n)
    rng = np.random.default_rng(1)
    if env_id == W3D:
        istep = rng.integers(0, t.n_steps, n).astype(np.int32)
        istep[:3] = t.clip_first_step[1:] - 1                         # the last step of every clip
    else:
        istep = (np.arange(n) % t.n_clips).astype(np.int32)
    pos = np.array([rng.integers(0, t.step_len[i]) for i in istep], np.int32)
    pos[:3] = t.step_len[istep[:3]] - 1
    og, oo = env.reset(inject=(istep, pos)), ora.reset(istep, pos)
    np.testing.assert_allclose(og, oo, rtol=2e-5, atol=2e-5)
    start = _clip_of(t, istep)
    wrapped = set()
    n_done = 0
    zero = np.zeros((n, env.act_dim), np.float32)
    for k in range(steps):
        prev = env.get_state()[2]
        og, rg, dg, _ = env.step(zero, inject=(istep, pos))
        oo, ro, do, _ = ora.step(zero, istep, pos)
        np.testing.assert_array_equal(dg, do, err_msg=f"done, step {k}")
        cg = env.get_state()[2]
        np.testing.assert_array_equal(cg[:, :3], np.array([[e.env.refs.i_step, e.env.refs.pos,
                                                             e.env.refs.count_steps_same_vel] for e in ora.envs]))
        ex = env.extras().cpu().numpy()
        # an env that did not end: the step's phase and desired velocity are those of the cursor it holds now
        for i in np.nonzero(~do)[0]:
            refs = ora.envs[i].env.refs
            i_s, p_s = int(cg[i, 0]), int(cg[i, 1])
            dv_o = refs.get_desired_walking_velocity_vector()[0]
            if env_id == W3D:
                assert ex[i, 6] == np.float32(p_s) / np.float32(t.step_len[i_s]), (k, i)
                assert ex[i, 5] == np.float32(dv_o), (k, i)
                assert bool(t.left_step[i_s]) == refs.is_step_left()
            else:
                hv = _host_des_vel(t, i_s, p_s)
                assert (np.isnan(hv) and np.isnan(ex[i, 5])) or hv == ex[i, 5], (k, i)
                assert (np.isnan(dv_o) and np.isnan(ex[i, 5])) or abs(dv_o - ex[i, 5]) <= 1e-6 * max(1.0, abs(dv_o))
            assert _clip_of(t, i_s) == start[i], (k, i)                   # never leaves its clip
        live = ~do
        wrap = live & ((cg[:, 0] < prev[:, 0]) if env_id == W3D else (cg[:, 1] == 0) & (prev[:, 1] > 0))
        wrapped |= set(start[wrap].tolist())
        start[do] = _clip_of(t, cg[do, 0])
        assert np.array_equal(np.isnan(og), np.isnan(oo))
        fin = np.isfinite(oo).all(axis=1)
        np.testing.assert_allclose(og[fin], oo[fin], rtol=2e-5, atol=2e-5)
        np.testing.assert_array_equal(np.signbit(rg), np.signbit(ro))
        assert np.abs(rg - ro).max() < 2e-5
        n_done += int(do.sum())
    assert n_done > 0
    assert wrapped == set(range(t.n_clips)), wrapped
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_id", [W3D, W165])
def test_playback_over_a_library(clip_dir, env_id):
    """kinematic playback with random RSI draws: every non-terminal step earns the maximal reward, across clip wraps,
    and the cursor never leaves the clip its episode started in"""
    paths = _w3d_paths(clip_dir) if env_id == W3D else _w165_paths(clip_dir)
    n, steps = 64, 1500
    cfg_kw = dict(ep_dur_max=1200)
    env = _gpu_env(env_id, n, paths, seed=3, **cfg_kw)
    t = env.spec.mocap
    cfg = env.cfg
    want = cfg.rew_scale * sum(cfg.rew_weights[:3]) + cfg.alive_bonus
    env.set_playback(True)
    env.reset()
    start = _clip_of(t, env.get_state()[2][:, 0])
    zeros = np.zeros((n, env.act_dim), np.float32)
    n_wrap = 0
    prev = env.get_state()[2][:, 0]
    for _ in range(steps):
        _, rew, done, _ = env.step(zeros)
        cur = env.get_state()[2][:, 0]
        if (~done).any():
            assert np.abs(rew[~done] - want).max() < 1e-6
        assert (_clip_of(t, cur[~done]) == start[~done]).all()
        n_wrap += int(((cur < prev) & ~done).sum())
        start[done] = _clip_of(t, cur[done])
        prev = cur
    assert n_wrap > 0 or env_id == W165
    env.set_playback(False)
    env.close()


def _mix64(x):
    x = (x + np.uint64(0x9E3779B97F4A7C15))
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def _host_draws(seed, n, resets, t):
    """the kernel's random RSI draw over a library, restated: (clip, step, sample) per env"""
    with np.errstate(over="ignore"):
        gid = np.arange(n, dtype=np.uint64)
        r = _mix64(_mix64(np.uint64(seed) ^ (gid * np.uint64(0xD1342543DE82EF95))) + np.uint64(resets))
        x = (_mix64(r ^ np.uint64(0x3C6EF372FE94F82B)) >> np.uint64(32)).astype(np.float64) * 2.0 ** -32
    w = np.asarray(t.clip_weight, np.float64)
    w = w / np.add.accumulate(w)[-1]
    cdf = np.add.accumulate(w) / np.add.accumulate(w)[-1]
    cdf[int(np.nonzero(w > 0)[0].max()):] = 1.0
    clip = np.searchsorted(cdf, x, side="right")
    first = t.clip_first_step[clip].astype(np.uint64)
    ns = (t.clip_first_step[clip + 1] - t.clip_first_step[clip]).astype(np.uint64)
    step = (first + (((r & np.uint64(0xFFFFFFFF)) * ns) >> np.uint64(32))).astype(np.int64)
    pos = (((r >> np.uint64(32)) * t.step_len[step].astype(np.uint64)) >> np.uint64(32)).astype(np.int64)
    return clip, step, pos


@pytest.mark.gpu
@pytest.mark.parametrize("weights", [None, [0.6, 0.0, 0.4]])
def test_sampler_at_65536_envs(clip_dir, weights):
    """start clips pass a chi-square test against the weights, steps are uniform within their clip, a zero-weight clip
    is never drawn; the draws are the restated counter-based draws exactly (cursor after the reset's next())"""
    n, resets, seed = 65536, 3, 17
    env = _gpu_env(W3D, n, _w3d_paths(clip_dir), weights, seed=seed)
    t = env.spec.mocap
    hist = np.zeros(t.n_clips, np.int64)
    step_hist = np.zeros(t.n_steps, np.int64)
    for r in range(resets):
        env.reset()
        cur = env.get_state()[2]
        clip, step, pos = _host_draws(seed, n, r, t)
        # the reset's next(): advance by one increment, per-clip wrap
        c = LibraryRefCursor(t, env.spec.model.nv)
        p1, s1 = pos + t.increment, step.copy()
        over = p1 - t.step_len[step] + 1 > 0
        for i in np.nonzero(over)[0]:
            c.init_random(int(step[i]), int(pos[i]))
            c.next()
            s1[i], p1[i] = c.i_step, c.pos
        np.testing.assert_array_equal(cur[:, 0], s1)
        np.testing.assert_array_equal(cur[:, 1], p1)
        hist += np.bincount(clip, minlength=t.n_clips)
        step_hist += np.bincount(step, minlength=t.n_steps)
    total = n * resets
    w = t.clip_weight
    pos_w = w > 0
    assert (hist[~pos_w] == 0).all()
    assert sps.chisquare(hist[pos_w], total * w[pos_w]).pvalue > ALPHA
    cf = t.clip_first_step
    for k in np.nonzero(pos_w)[0]:
        h = step_hist[cf[k]:cf[k + 1]]
        assert sps.chisquare(h).pvalue > ALPHA, (k, h)
    env.close()


@pytest.mark.gpu
def test_clip_stats_equal_a_host_replay(clip_dir):
    """per-clip episodes, summed lengths, timeouts and falls + blow-ups equal a replay of the run's done flags, start
    clips and episode lengths, exactly; the totals equal the 20 statistics"""
    n, steps = 512, 300
    env = _gpu_env(W3D, n, _w3d_paths(clip_dir), seed=4, early_termination=True, ep_dur_max=60)
    t = env.spec.mocap
    with pytest.raises(lib.DrlError):
        _gpu_env(W3D, 4).clip_stats()
    acts = _acts(n, env.act_dim, steps, 2)
    env.reset_tensor()
    start = _clip_of(t, env.get_state()[2][:, 0])
    eps, lens, tos = (np.zeros(t.n_clips, np.int64) for _ in range(3))
    for k in range(steps):
        ep_dur = env.get_state()[2][:, 3]
        d = env.step_tensor(acts[k])[2].cpu().numpy().astype(bool)
        ln = ep_dur + 1
        np.add.at(eps, start[d], 1)
        np.add.at(lens, start[d], ln[d])
        np.add.at(tos, start[d & (ln >= 60)], 1)
        start[d] = _clip_of(t, env.get_state()[2][d, 0])
    cs = env.clip_stats()
    assert set(cs) == {"episodes", "ep_len_sum", "falls", "timeouts", "blowups"}
    np.testing.assert_array_equal(cs["episodes"], eps)
    np.testing.assert_array_equal(cs["ep_len_sum"], lens)
    np.testing.assert_array_equal(cs["falls"] + cs["timeouts"] + cs["blowups"], eps)
    st = env.stats()
    assert cs["timeouts"].sum() == st["timeouts"] and cs["falls"].sum() == st["falls"]
    assert cs["blowups"].sum() == st["blowups"] and eps.sum() == st["episodes"] and lens.sum() == st["ep_len_sum"]
    np.testing.assert_array_equal(cs["timeouts"] + cs["blowups"] >= tos, True)
    assert (eps > 0).all() and cs["falls"].sum() > 0 and cs["timeouts"].sum() > 0
    assert env.mocap_clips()[1]["path"].endswith("ramp4.mat") and env.mocap_clips()[1]["steps"] == 4
    env.close()


@pytest.mark.gpu
def test_adaptive_rsi_on_a_library(clip_dir):
    """failure-weighted RSI over a library with non-default weights: the table's u is the library's base draw and the
    decayed counts equal a float64 replay, exactly"""
    n, steps, H = 384, 250, 40
    env = _gpu_env(W3D, n, _w3d_paths(clip_dir), [0.5, 0.2, 0.3], seed=3, early_termination=True, adaptive_rsi=0.5,
                   adaptive_rsi_halflife=H)
    t = env.spec.mocap
    acts = _acts(n, env.act_dim, steps, 8)
    env.reset_tensor()
    tab = env.adaptive_rsi_table()
    want = adaptive_rsi_bins(t.step_len, ADAPTIVE_RSI_BIN_STEPS * t.increment, t.clip_first_step, t.clip_weight)
    np.testing.assert_array_equal(tab["u"], want["u"])
    np.testing.assert_allclose(tab["prob"], tab["u"], rtol=1e-12)
    nb = len(tab["u"])
    s, f = np.zeros(nb), np.zeros(nb)
    rho = 2.0 ** (-1.0 / H)
    bins = tab["env_bin"]
    n_ep = 0
    for k in range(steps):
        ep_dur = env.get_state()[2][:, 3]
        d = env.step_tensor(acts[k])[2].cpu().numpy().astype(bool)
        sm = np.array(env.get_attr("ep_len_smoothed"), np.float32)
        ended = d & (bins >= 0)
        diff = ended & (np.float32(ep_dur + 1) < sm * np.float32(0.75))
        s = rho * s + np.bincount(bins[ended], minlength=nb).astype(np.float64)
        f = rho * f + np.bincount(bins[diff], minlength=nb).astype(np.float64)
        n_ep += int(ended.sum())
        tab = env.adaptive_rsi_table()
        np.testing.assert_array_equal(tab["started"], s, err_msg=f"step {k}")
        np.testing.assert_array_equal(tab["difficult"], f, err_msg=f"step {k}")
        bins = tab["env_bin"]
    assert n_ep > 100
    # every start bin lies in the clip of its episode's cursor
    cur = env.get_state()[2][:, 0]
    np.testing.assert_array_equal(_clip_of(t, tab["step"][bins]), _clip_of(t, cur))
    env.close()


@pytest.mark.gpu
def test_graph_path_and_bit_reproducibility(clip_dir):
    """the CUDA-graph VecNormalize path over a library: two identical runs agree bit for bit, clip counts included,
    and the library setters keep their errors: no clip change while failure-weighted RSI is on"""
    from drloco_b200.vec_env import vec_env
    n, steps = 1024, 120
    runs = []
    for _ in range(2):
        v = vec_env(W3D, num_envs=n, seed=8, mocap_path=_w3d_paths(clip_dir), clip_weights=[1, 1, 2],
                    cfg=EnvConfig(env_id=W3D, early_termination=True, ep_dur_max=80))
        assert v.use_graph
        rng = np.random.default_rng(5)
        obs = [v.reset()]
        for _ in range(steps):
            o, r, d, _ = v.step(rng.uniform(-1, 1, (n, v.venv.act_dim)).astype(np.float32))
            obs += [o, r, d]
        assert v.use_graph
        runs.append((np.concatenate([np.asarray(x, np.float64).ravel() for x in obs]), v.venv.clip_stats(),
                     v.venv.get_state()[2]))
        v.close()
    np.testing.assert_array_equal(runs[0][0], runs[1][0])
    np.testing.assert_array_equal(runs[0][2], runs[1][2])
    for k in runs[0][1]:
        np.testing.assert_array_equal(runs[0][1][k], runs[1][1][k])
    assert runs[0][1]["episodes"].sum() > 0


@pytest.mark.gpu
def test_abi_state_errors_and_evaluation_guard(clip_dir):
    L = lib.load()
    env = _gpu_env(W3D, 8, _w3d_paths(clip_dir), adaptive_rsi=0.5)
    t = env.spec.mocap
    first = np.ascontiguousarray(t.clip_first_step, np.int32)
    w = np.ones(t.n_clips)
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    assert L.drl_set_mocap_clips(env._handle, t.n_clips, p(first), p(w)) == -3          # DRL_ERR_STATE: ARS on
    lib.check(L.drl_set_adaptive_rsi(env._handle, 0.0, 2000, 40), "drl_set_adaptive_rsi")
    lib.check(L.drl_set_mocap_clips(env._handle, t.n_clips, p(first), p(w)), "drl_set_mocap_clips")
    for bad_first, bad_w in (([0, 3, 7, 8], w), ([1, 3, 7, 9], w), ([0, 1, 7, 9], w), ([0, 7, 3, 9], w),
                             (first, np.array([1.0, -1.0, 1.0])), (first, np.zeros(3)),
                             (first, np.array([1.0, np.nan, 1.0]))):
        bf = np.ascontiguousarray(bad_first, np.int32)
        bw = np.ascontiguousarray(bad_w, np.float64)
        assert L.drl_set_mocap_clips(env._handle, 3, p(bf), p(bw)) == -1, (bad_first, bad_w)
    out = np.zeros((t.n_clips, 5), np.int64)
    import torch
    dev_out = torch.zeros(t.n_clips, 5, dtype=torch.int64, device="cuda")
    lib.check(L.drl_get_clip_stats(env._handle, C.c_void_p(dev_out.data_ptr()), None), "drl_get_clip_stats")
    torch.cuda.synchronize()
    assert (dev_out.cpu().numpy() == out).all()
    # one clip again: the counters go away
    one = np.array([0, t.n_steps], np.int32)
    lib.check(L.drl_set_mocap_clips(env._handle, 1, p(one), p(np.ones(1))), "drl_set_mocap_clips")
    assert L.drl_get_clip_stats(env._handle, C.c_void_p(dev_out.data_ptr()), None) == -3
    env.close()
    # evaluation starts from the first eval_n_times steps of clip 0: a short clip 0 is refused
    env = _gpu_env(W3D, 4, _w3d_paths(clip_dir))
    with pytest.raises(ValueError, match="eval_n_times"):
        env.env_method("activate_evaluation")
    env.close()
    env = _gpu_env(W3D, 4, [None, str(clip_dir / "s2.npz")], eval_n_times=5)
    env.env_method("activate_evaluation")
    env.reset()
    assert (env.get_state()[2][:, 0] < 30).all()
    env.close()
    # a wrap-mode table of several steps cannot be stepped as one clip
    env = _gpu_env(W165, 4, _w165_paths(clip_dir))
    one = np.array([0, 2], np.int32)
    assert L.drl_set_mocap_clips(env._handle, 1, p(one), p(np.ones(1))) == -1             # a wrap clip is one step
    env.close()
