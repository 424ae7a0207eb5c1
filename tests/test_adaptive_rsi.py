"""Opt-in failure-weighted reference state initialisation (EnvConfig(adaptive_rsi=lambda), drl_set_adaptive_rsi).

The mocap is cut into bins of at most 20 control steps of reference motion inside each mocap step.  Per bin the env
keeps decayed float64 counts of the episodes that started there (s) and of those that were difficult by Monitor's rule
(f).  A random RSI draw takes, with probability lambda, a bin from q_b ~ u_b (f_b + 1) / (s_b + 2) and a sample uniform
in it (u_b: the bin's probability under the reference's uniform draw), and otherwise the uniform draw, bit for bit.

The float64 model of the table below (bins, decay, mixture) is the reference the GPU results are held against."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
from scipy import stats as sps

from drloco_b200 import lib
from drloco_b200.config import EnvConfig
from drloco_b200.vec_env import ADAPTIVE_RSI_BIN_STEPS, adaptive_rsi_bins
from drloco_b200.walkers import make_spec

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W3D, W165 = "StraightMimicWalker", "MimicWalker165cm65kg"
ALPHA = 1e-3        # significance level of the chi-square tests (fixed seeds: the outcome is deterministic)


# --------------------------------------------------------------------------------------------------------------------
# float64 model of the table
# --------------------------------------------------------------------------------------------------------------------
def decay(x, dx, halflife):
    """one update of a count: x <- rho x + dx, rho = 2^(-1/H), rounded in that order (as the update kernel)"""
    rho = 2.0 ** (-1.0 / halflife)
    return rho * x + dx


def mixture(u, started, difficult, lam):
    """(q, p): the weighted distribution and the full mixture p = (1 - lambda) u + lambda q"""
    w = u * ((difficult + 1.0) / (started + 2.0))
    q = w / w.sum()
    return q, (1.0 - lam) * u + lam * q


def _bins(env_id):
    t = make_spec(EnvConfig(env_id=env_id)).mocap
    return t, adaptive_rsi_bins(t.step_len, ADAPTIVE_RSI_BIN_STEPS * t.increment)


@pytest.mark.parametrize("env_id,n_bins,width", [(W3D, 210, 40), (W165, 300, 100)])
def test_bin_table_covers_every_sample_once(env_id, n_bins, width):
    t, b = _bins(env_id)
    assert len(b["u"]) == n_bins and int(b["width"].max()) == width
    hits = [np.zeros(int(n), np.int32) for n in t.step_len]
    for s, f, w in zip(b["step"], b["first"], b["width"]):
        assert 0 < w <= width and f + w <= t.step_len[s]          # inside its step: no bin straddles two
        hits[s][f:f + w] += 1
    assert all((h == 1).all() for h in hits)
    assert np.isclose(b["u"].sum(), 1.0, rtol=0, atol=1e-12)
    # u is the reference's draw: a uniform step, then a uniform sample in it
    for s in range(t.n_steps):
        assert np.isclose(b["u"][b["step"] == s].sum(), 1.0 / t.n_steps, rtol=1e-12)


def test_model_known_answers():
    _, b = _bins(W3D)
    u, n = b["u"], len(b["u"])
    zero = np.zeros(n)
    # an empty table is the reference distribution, whatever lambda
    for lam in (0.0, 0.3, 1.0):
        q, p = mixture(u, zero, zero, lam)
        np.testing.assert_allclose(q, u, rtol=1e-13)
        np.testing.assert_allclose(p, u, rtol=1e-13)
    # one saturated bin k (every episode started there was difficult), all others untouched: rate_k = (N + 1) / (N + 2)
    # against 1/2, so q_k / q_j = (u_k / u_j) * 2 (N + 1) / (N + 2)
    k, N = 17, 1000.0
    s, f = zero.copy(), zero.copy()
    s[k] = f[k] = N
    q, p = mixture(u, s, f, 1.0)
    for j in (0, 5, n - 1):
        assert np.isclose(q[k] / q[j], (u[k] / u[j]) * 2.0 * (N + 1.0) / (N + 2.0), rtol=1e-13)
    np.testing.assert_array_equal(p, q)                           # lambda = 1: the weighted part alone
    _, p_small = mixture(u, s, f, 1e-9)                           # lambda -> 0: the reference distribution
    np.testing.assert_allclose(p_small, u, rtol=1e-8)
    _, p_half = mixture(u, s, f, 0.5)
    np.testing.assert_allclose(p_half, 0.5 * u + 0.5 * q, rtol=1e-15)
    # the half-life: H updates without new episodes halve a count
    x = 8.0
    for _ in range(2000):
        x = decay(x, 0.0, 2000)
    assert np.isclose(x, 4.0, rtol=1e-12)


def test_config_default_and_validation():
    c = EnvConfig()
    assert c.adaptive_rsi == 0.0 and c.adaptive_rsi_halflife == 2000
    assert EnvConfig(adaptive_rsi=0.5, adaptive_rsi_halflife=100).adaptive_rsi == 0.5
    EnvConfig(adaptive_rsi=1)
    for bad in (-0.1, 1.5, float("nan"), "0.5", True, None):
        with pytest.raises(ValueError):
            EnvConfig(adaptive_rsi=bad)
    for bad in (0, -5, 2.5, 2 ** 31, True):
        with pytest.raises(ValueError):
            EnvConfig(adaptive_rsi=0.5, adaptive_rsi_halflife=bad)


@pytest.fixture(scope="module")
def built_lib():
    if not os.path.exists(lib.LIB_PATH):
        sys.path.insert(0, REPO)
        import __graft_entry__
        __graft_entry__.build()
    return lib.load()


def test_abi_argument_errors_without_a_device(built_lib):
    L = built_lib
    assert L.drl_set_adaptive_rsi(None, 0.5, 2000, 40) == -1          # DRL_ERR_INVALID
    assert b"null env" in L.drl_last_error()
    buf = (C.c_double * 4)()
    assert L.drl_get_adaptive_rsi(None, C.cast(buf, C.c_void_p), None, None, None, None) == -1
    assert b"null env" in L.drl_last_error()
    assert L.drl_set_adaptive_rsi_counts(None, C.cast(buf, C.c_void_p), C.cast(buf, C.c_void_p)) == -1
    assert b"null argument" in L.drl_last_error()


# --------------------------------------------------------------------------------------------------------------------
# GPU
# --------------------------------------------------------------------------------------------------------------------
def _gpu_env(env_id, n, **kw):
    from drloco_b200.vec_env import B200MimicVecEnv
    seed = kw.pop("seed", 5)
    return B200MimicVecEnv(env_id, num_envs=n, cfg=EnvConfig(env_id=env_id, **kw), seed=seed)


def _set(env, lam, halflife=2000):
    bs = ADAPTIVE_RSI_BIN_STEPS * env.spec.mocap.increment
    lib.check(lib.load().drl_set_adaptive_rsi(env._handle, lam, halflife, bs), "drl_set_adaptive_rsi")


MONITOR = ("mean_ep_pos_rew_smoothed", "mean_ep_vel_rew_smoothed", "mean_ep_com_rew_smoothed", "mean_reward_smoothed",
           "ep_ret_smoothed", "ep_len_smoothed", "moved_distance", "mean_abs_ep_torque_smoothed")


def _run_tensor(env, acts, inject=None):
    """reset + steps on the tensor path; every output of the run"""
    import torch
    outs = [env.reset_tensor(inject=inject).clone()]
    for a in acts:
        o, r, d = env.step_tensor(a, inject)
        outs += [o.clone(), r.clone(), d.clone(), env.terminal_obs.clone()]
    q, v, c = env.get_state()
    return dict(outs=torch.cat([x.float().flatten() for x in outs]).cpu().numpy(), q=q, v=v, c=c,
                stats=env.stats(), extras=env.extras().cpu().numpy(), ring=env.episode_records(),
                monitor={k: env.get_attr(k) for k in MONITOR})


def _assert_runs_equal(a, b):
    for k in ("outs", "q", "v", "c", "extras"):
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert a["stats"] == b["stats"]
    assert a["monitor"] == b["monitor"]
    # the episode ring: slots are taken in the order in which thread blocks finish, so compare the records as a set
    rec = lambda r: sorted(zip(*(r[k].tolist() for k in sorted(r))))   # noqa: E731
    assert rec(a["ring"]) == rec(b["ring"])


def _acts(n, act_dim, steps, seed):
    import torch
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.rand(steps, n, act_dim, device="cuda", generator=g) * 2 - 1


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,integrator,actuation", [(W3D, "rk4", "torque"), (W3D, "euler", "torque"),
                                                         (W165, "rk4", "torque"), (W3D, "rk4", "pd")])
def test_off_is_the_parent(env_id, integrator, actuation):
    """adaptive_rsi = 0 (never enabled), and enabled then set back to lambda = 0, give every output of a fresh env,
    bit for bit; the run with the option on starts its episodes elsewhere"""
    n, steps = 256, 250
    kw = dict(integrator=integrator, seed=9)
    if actuation == "pd":
        kw.update(actuation="pd", pd_kp=200.0, pd_kv=5.0)
    acts = _acts(n, make_spec(EnvConfig(env_id=env_id)).act_dim, steps, 4)

    def run(before=None, **extra):
        env = _gpu_env(env_id, n, **kw, **extra)
        if before:
            before(env)
        out = _run_tensor(env, acts)
        env.close()
        return out
    fresh = run()
    _assert_runs_equal(run(adaptive_rsi=0.0), fresh)
    _assert_runs_equal(run(before=lambda e: (_set(e, 0.7), _set(e, 0.0))), fresh)
    on = run(adaptive_rsi=1.0)
    assert not np.array_equal(on["c"], fresh["c"])


def _difficult(ep_len, smoothed):
    """Monitor's bit (monitor_wrapper.py:123-124) in float32, as the kernel evaluates it"""
    return np.float32(ep_len) < np.float32(smoothed) * np.float32(0.75)


@pytest.mark.gpu
@pytest.mark.parametrize("env_id,integrator", [(W3D, "rk4"), (W3D, "euler"), (W165, "rk4")])
def test_counts_equal_a_float64_replay(env_id, integrator):
    """per-env start bins and done after every step, the difficult bit recomputed from ep_len_smoothed: the decayed
    counts equal a float64 replay of the same operations in the same order, exactly.  early_termination makes the
    episode lengths vary enough under random actions for some episodes to be difficult."""
    import torch
    n, steps, H = 384, 300, 40
    env = _gpu_env(env_id, n, seed=3, integrator=integrator, early_termination=True, adaptive_rsi=0.5,
                   adaptive_rsi_halflife=H)
    acts = _acts(n, env.act_dim, steps, 8)
    env.reset_tensor()
    tab = env.adaptive_rsi_table()
    nb = len(tab["u"])
    s, f = np.zeros(nb), np.zeros(nb)
    bins = tab["env_bin"]
    assert (bins >= 0).all()
    np.testing.assert_allclose(tab["prob"], tab["u"], rtol=1e-12)
    n_ep = n_diff = 0
    for k in range(steps):
        ep_dur = env.get_state()[2][:, 3]
        d = env.step_tensor(acts[k])[2].cpu().numpy().astype(bool)
        sm = np.array(env.get_attr("ep_len_smoothed"), np.float32)
        ended = d & (bins >= 0)
        diff = ended & _difficult(ep_dur + 1, sm)
        s = decay(s, np.bincount(bins[ended], minlength=nb).astype(np.float64), H)
        f = decay(f, np.bincount(bins[diff], minlength=nb).astype(np.float64), H)
        n_ep += int(ended.sum())
        n_diff += int(diff.sum())
        tab = env.adaptive_rsi_table()
        np.testing.assert_array_equal(tab["started"], s, err_msg=f"started, step {k}")
        np.testing.assert_array_equal(tab["difficult"], f, err_msg=f"difficult, step {k}")
        nb_new = tab["env_bin"]
        np.testing.assert_array_equal(nb_new[~d], bins[~d])            # a running episode keeps its bin
        assert (nb_new[d] >= 0).all()                                   # every auto-reset is a random draw
        bins = nb_new
    assert n_ep > 200 and 0 < n_diff < n_ep
    _, p = mixture(tab["u"], s, f, 0.5)
    np.testing.assert_allclose(tab["prob"], p, rtol=1e-12)
    env.close()
    torch.cuda.synchronize()


def _drawn_positions(spec, table, cursor):
    """the RSI sample of every env, recovered from its start bin and the cursor after the reset's `next()`"""
    t = spec.mocap
    b = table["env_bin"]
    step = table["step"][b]
    i, pos = cursor[:, 0], cursor[:, 1]
    same = i == step
    p0 = np.where(same, pos - t.increment, pos + t.step_len[step] - 1 - t.increment)
    return b, p0


@pytest.mark.gpu
def test_sampler_matches_the_mixture():
    """65 536 envs, a skewed table pinned with set_adaptive_rsi_table, several resets: the start-bin histogram passes
    a chi-square test against the float64 mixture, every sample lies in its bin, and the offsets inside full-width
    bins pass a pooled chi-square test for uniformity; with lambda = 1 and one favoured bin its share matches q"""
    n, resets = 65536, 4
    env = _gpu_env(W3D, n, seed=17, adaptive_rsi=0.5)
    spec = env.spec
    tab = env.adaptive_rsi_table()
    u = tab["u"]
    nb = len(u)
    rng = np.random.default_rng(2)
    s = np.full(nb, 100.0)
    f = np.floor(rng.uniform(0, 1, nb) ** 3 * 100.0)
    env.set_adaptive_rsi_table(s, f)
    _, p = mixture(u, s, f, 0.5)
    np.testing.assert_allclose(env.adaptive_rsi_table()["prob"], p, rtol=1e-12)
    hist = np.zeros(nb, np.int64)
    off = np.zeros(ADAPTIVE_RSI_BIN_STEPS * spec.mocap.increment, np.int64)
    for _ in range(resets):
        env.reset()
        tab = env.adaptive_rsi_table()
        b, p0 = _drawn_positions(spec, tab, env.get_state()[2])
        assert (b >= 0).all()
        first, width = tab["first"][b], tab["width"][b]
        assert ((p0 >= first) & (p0 < first + width)).all()
        hist += np.bincount(b, minlength=nb)
        full = width == len(off)
        off += np.bincount(p0[full] - first[full], minlength=len(off))
        np.testing.assert_array_equal(tab["started"], s)                # resets alone count nothing
    total = n * resets
    assert sps.chisquare(hist, total * p).pvalue > ALPHA
    assert sps.chisquare(off).pvalue > ALPHA
    # lambda = 1, one favoured bin
    k = 77
    s1, f1 = np.full(nb, 1e4), np.zeros(nb)
    f1[k] = 1e4
    _set(env, 1.0)
    env.set_adaptive_rsi_table(s1, f1)
    q, p1 = mixture(u, s1, f1, 1.0)
    np.testing.assert_allclose(env.adaptive_rsi_table()["prob"], p1, rtol=1e-12)
    env.reset()
    b = env.adaptive_rsi_table()["env_bin"]
    share = float(np.mean(b == k))
    assert abs(share - q[k]) < 5.0 * np.sqrt(q[k] * (1 - q[k]) / n), (share, q[k])
    assert q[k] > 0.9
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["eval", "speed", "inject", "set_state"])
def test_excluded_starts_are_not_counted_and_draw_as_without_the_option(mode):
    """evaluation mode, speed profile, injected draws: the start bin stays -1, the counts do not move, and every output
    equals the option-off run; a state set with set_state uncounts the running episodes"""
    n, steps = 128, 200
    acts = _acts(n, 8, steps, 6)
    rng = np.random.default_rng(0)
    t = make_spec(EnvConfig(env_id=W3D)).mocap
    istep = rng.integers(0, t.n_steps, n).astype(np.int32)
    pos = np.array([rng.integers(0, t.step_len[i]) for i in istep], np.int32)
    if mode == "set_state":
        env = _gpu_env(W3D, n, seed=12, adaptive_rsi=1.0)
        env.reset()
        assert (env.adaptive_rsi_table()["env_bin"] >= 0).all()
        env.set_state(*env.get_state())
        assert (env.adaptive_rsi_table()["env_bin"] == -1).all()
        for a in acts[:20]:
            env.step_tensor(a)
        assert (env.adaptive_rsi_table()["started"] == 0).all()
        env.close()
        return
    runs = []
    for lam in (0.0, 1.0):
        env = _gpu_env(W3D, n, seed=12, adaptive_rsi=lam)
        inject = None
        if mode == "eval":
            env.env_method("activate_evaluation")
        elif mode == "speed":
            env.activate_speed_control((0.8, 1.2), 2)
        elif mode == "inject":
            inject = (istep, pos)
        runs.append(_run_tensor(env, acts, inject))
        if lam > 0:
            tab = env.adaptive_rsi_table()
            assert (tab["env_bin"] == -1).all()
            assert (tab["started"] == 0).all() and (tab["difficult"] == 0).all()
            np.testing.assert_allclose(tab["prob"], tab["u"], rtol=1e-12)
        env.close()
    assert runs[0]["stats"]["episodes"] > 0
    _assert_runs_equal(*runs)


@pytest.mark.gpu
def test_two_identical_runs_are_bit_identical():
    n, steps = 512, 250
    acts = _acts(n, 8, steps, 3)
    runs, tabs = [], []
    for _ in range(2):
        env = _gpu_env(W3D, n, seed=21, adaptive_rsi=0.5, adaptive_rsi_halflife=50)
        runs.append(_run_tensor(env, acts))
        tabs.append(env.adaptive_rsi_table())
        env.close()
    _assert_runs_equal(*runs)
    for k in tabs[0]:
        np.testing.assert_array_equal(tabs[0][k], tabs[1][k], err_msg=k)
    assert tabs[0]["started"].sum() > 0


@pytest.mark.gpu
def test_vecnormalize_graph_path_equals_the_tensor_path():
    import torch
    from drloco_b200.vec_env import B200VecNormalize
    n, steps = 256, 250
    rng = np.random.default_rng(6)
    acts = rng.uniform(-1, 1, (steps, n, 8)).astype(np.float32)
    res, tabs = [], []
    for graph in (True, False):
        env = _gpu_env(W3D, n, seed=13, adaptive_rsi=0.5, adaptive_rsi_halflife=50)
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
            l0 = env.launches + vn.launches
            for a in acts:
                o, r, d = vn.step_tensor(torch.from_numpy(a).cuda())
                outs.append((o.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy().astype(bool)))
            assert env.launches + vn.launches - l0 == 3 * steps      # step kernel, table update, statistics kernel
        res.append(outs)
        tabs.append(env.adaptive_rsi_table())
        env.close()
    assert any(d.any() for _, _, d in res[0]) and tabs[0]["started"].sum() > 0
    for k in tabs[0]:
        np.testing.assert_array_equal(tabs[0][k], tabs[1][k], err_msg=k)
    for (o1, r1, d1), (o2, r2, d2) in zip(*res):
        np.testing.assert_array_equal(o1, o2)
        np.testing.assert_array_equal(r1, r2)
        np.testing.assert_array_equal(d1, d2)


@pytest.mark.gpu
def test_call_order_and_argument_errors():
    import torch
    from drloco_b200 import cabi
    L = lib.load()
    env = _gpu_env(W3D, 8)                                            # option off (default)
    buf = torch.zeros(300, dtype=torch.float64, device="cuda")
    assert L.drl_get_adaptive_rsi(env._handle, C.c_void_p(buf.data_ptr()), None, None, None, None) == -3
    assert b"never enabled" in L.drl_last_error()
    h = np.zeros(210)
    hp = h.ctypes.data_as(C.c_void_p)
    assert L.drl_set_adaptive_rsi_counts(env._handle, hp, hp) == -3
    with pytest.raises(lib.DrlError):
        env.adaptive_rsi_table()
    with pytest.raises(lib.DrlError):
        env.set_adaptive_rsi_table(h, h)
    for lam, hl, bs in ((-0.1, 10, 40), (1.01, 10, 40), (float("nan"), 10, 40), (0.5, 0, 40), (0.5, 10, 0)):
        assert L.drl_set_adaptive_rsi(env._handle, lam, hl, bs) == -1, (lam, hl, bs)
    assert L.drl_set_adaptive_rsi(env._handle, 0.0, 10, 40) == 0        # off stays off: no table yet
    assert L.drl_get_adaptive_rsi(env._handle, C.c_void_p(buf.data_ptr()), None, None, None, None) == -3
    assert L.drl_set_adaptive_rsi(env._handle, 0.5, 10, 40) == 0
    assert L.drl_get_adaptive_rsi(env._handle, C.c_void_p(buf.data_ptr()), None, None, None, None) == 0
    bad = np.zeros(210)
    bad[3] = 1.0                                                       # difficult > started
    assert L.drl_set_adaptive_rsi_counts(env._handle, hp, bad.ctypes.data_as(C.c_void_p)) == -1
    with pytest.raises(lib.DrlError, match="stale"):
        env._upload_mocap()                                             # on: the bins would go stale
    assert L.drl_set_adaptive_rsi(env._handle, 0.0, 10, 40) == 0
    env._upload_mocap()                                                 # off again: allowed
    env.close()
    env = _gpu_env(W3D, 8, adaptive_rsi=0.5)
    with pytest.raises(ValueError):
        env.set_adaptive_rsi_table(np.zeros(3), np.zeros(3))
    env.close()
    spec = make_spec()
    cfg = cabi.DrlConfig()
    cfg.num_envs, cfg.device, cfg.frame_skip, cfg.obs_dim, cfg.act_dim, cfg.ctrl_freq = 8, 0, 5, 29, 8, 200.0
    hd = C.c_void_p()
    assert L.drl_create(C.byref(cfg), C.byref(hd)) == 0
    assert L.drl_set_adaptive_rsi(hd, 0.5, 10, 40) == -3                # DRL_ERR_STATE: no model / mocap yet
    cm = cabi.pack_model(spec.model)
    assert L.drl_upload_model(hd, C.byref(cm)) == 0
    assert L.drl_set_adaptive_rsi(hd, 0.5, 10, 40) == -3                # no mocap yet
    assert L.drl_destroy(hd) == 0
