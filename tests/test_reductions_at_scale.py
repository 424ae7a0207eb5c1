"""The reduction and bookkeeping kernels at production and ragged shapes, against float64 references.

Covered: the statistics epilogue of the step kernel (csrc/mimic_step.cu, the two-level fixed-order sum behind the
VecNormalize batch moments and ``env.stats()``), the VecNormalize kernels of csrc/vecnorm.cu (moments, merge +
normalisation with its ``stats_sync_every`` cycle, terminal-row compaction), the radix-select median behind Monitor's
``median_abs_torque_smoothed`` past its shared-memory staging capacity, and the wrap of the episode ring.

Every tolerance below is derived from the arithmetic, with u64 = 2^-53 and u32 = 2^-24 the unit roundoffs:

* A float64 sum of terms x_i, in any order, whose summation tree is at most ``depth`` additions deep is off the exact
  sum by at most depth * u64 * sum|x_i| (first order).  The step kernel adds a term at most
  ``_epilogue_depth(epb, ngroups)`` times; numpy's pairwise sum at most ``REF_DEPTH`` times.
* Batch moments: with c such a depth bound, |mean error| <= c u64 E|x| and the one-pass variance
  ``sumsq/n - mean^2`` (the kernel's) is off the two-pass ``np.var`` by at most (3c + 4) u64 E[x^2]: the two sums
  contribute c u64 E[x^2] and 2 |mean| c u64 E|x| <= 2 c u64 E[x^2] (Cauchy-Schwarz), the subtraction one rounding, the
  reference's own two-pass variance c u64 E[(x-mean)^2].  Relative to the variance this is (3c + 4) u64 (1 + mean^2/var):
  a column with |mean|/std = 1e3 loses six decimal digits to the one-pass formula.
* Running statistics (Chan merge): the merged mean is a convex combination of the batch means, so its error is the
  largest batch-mean error plus about 4 u64 |mean| of rounding per merge.  The merged variance also carries the error of
  the between-batch term delta^2 (at most 8 c u64 E[x^2], with delta and its error bounded as above) and about 24 u64
  E[x^2] of rounding per merge.  ``_RmsBound`` accumulates these bounds; they come to about 1e-12 relative.
* Normalisation (float32 on the device): the kernel computes fl(fl(x - fl(mean)) * fl(1/sqrt(var + eps))).  Against the
  float64 z = (x - mean)/sqrt(var + eps) of the same statistics that is at most
  u32 (inv |mean| + 3 |z|) (1 + 1%) off (rounding of the mean, the subtraction, the inverse square root, the product;
  ``_norm_ref``).  Clipping is 1-Lipschitz and the clip bounds are float32 values, so the bound holds after clipping.
  Where the statistics themselves carry an error (dmean, dvar) the bound grows by inv dmean + |z| dvar / (2 (var+eps)).
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from drloco_b200.config import EnvConfig  # noqa: E402

W3D, W165 = "StraightMimicWalker", "MimicWalker165cm65kg"
LANES = {W3D: 16, W165: 32}                    # lanes per environment (G) of each walker's step kernel
STAT_GROUP = 16                                # kStatGroup of csrc/mimic_step.cu
# shared-memory staging capacity of the median (floats): EnvSmem<G> in csrc/fd_tree.cuh, from S[0][0] up to Mt, minus
# the 256 histogram bins (mimic_step.cu, group_median's caller)
MEDIAN_CAP = {16: 704, 32: 1536}
U64, U32 = 2.0 ** -53, 2.0 ** -24
REF_DEPTH = 40       # numpy's pairwise sum (8 partials over blocks of 128, then halving: < 30 levels at 2^16 rows),
#                      plus the roundings of the mean / variance formulas

# (walker, num_envs, CTA threads): single-block grid, last group of one block, 8-way loop and remainder loop of the
# final sum in the same call, padding environments for G = 16 and G = 32, grids above 2048 blocks
EPILOGUE_CASES = [
    (W3D, 1, 128),
    (W3D, 129, 128),
    (W3D, 4097, 128),
    (W3D, 4096, 96),
    (W3D, 65535, 32),
    (W3D, 65536, 128),
    (W165, 1001, 96),
    (W165, 16383, 128),
]


def _launch_shape(walker, n, block):
    """(G, environments per block, grid, padding environments, groups of STAT_GROUP blocks, blocks in the last group)"""
    G = LANES[walker]
    epb = block // G
    grid = -(-n // epb)
    ngroups = -(-grid // STAT_GROUP)
    return G, epb, grid, grid * epb - n, ngroups, grid - (ngroups - 1) * STAT_GROUP


def _epilogue_depth(epb, ngroups):
    """additions a term passes through in the step kernel's sum: block row (epb - 1), group row (16 rows into 4
    partials, then 2 levels), final row (ngroups // 8 + 7 rows into 8 partials, then 3 levels)"""
    return (epb - 1) + (4 + 2) + (ngroups // 8 + 7 + 3)


def _moments_depth(n, d):
    """the same for csrc/vecnorm.cu::vecnorm_moments_kernel: the rows one thread walks, then at most 256 shared and 592
    global atomic additions (one per block)"""
    blocks = min(max(1, -(-n * d // 2048)), 592)
    step = (blocks * 256 // d) * d
    return -(-n * d // step) + 256 + blocks


# ---------------------------------------------------------------------------------------------------------------------
# float64 reference helpers
# ---------------------------------------------------------------------------------------------------------------------
class _RmsBound:
    """running error bound of device statistics against a float64 RunningMeanStd fed the same batches (module
    docstring): per column, the largest batch-moment errors plus the rounding of every merge."""

    def __init__(self, depth, shape):
        self.c = depth + REF_DEPTH
        self.bmean = np.zeros(shape)          # largest batch-mean error bound so far
        self.sq = np.ones(shape)              # largest E[x^2] so far (the initial statistics: mean 0, var 1)
        self.merges = 0

    def add(self, x):
        x = np.asarray(x, np.float64)
        self.bmean = np.maximum(self.bmean, self.c * U64 * np.abs(x).mean(axis=0))
        self.sq = np.maximum(self.sq, (x * x).mean(axis=0))
        self.merges += 1

    def tols(self, ref):
        """(mean, variance) bounds against the float64 reference statistics ``ref``"""
        self.sq = np.maximum(self.sq, np.asarray(ref.var) + np.asarray(ref.mean) ** 2)
        tol_m = self.bmean + 4 * self.merges * U64 * np.abs(ref.mean)
        return tol_m, ((11 * self.c + 4) + 24 * self.merges) * U64 * self.sq

    def check(self, mean, var, ref, what):
        tol_m, tol_v = self.tols(ref)
        assert np.all(np.abs(mean - ref.mean) <= tol_m), f"{what} mean: {np.max(np.abs(mean - ref.mean) / tol_m)}"
        assert np.all(np.abs(var - ref.var) <= tol_v), f"{what} var: {np.max(np.abs(var - ref.var) / tol_v)}"
        return tol_m, tol_v


def _norm_ref(x, mean, var, eps, clip, dmean=0.0, dvar=0.0):
    """float64 clip((x - mean)/sqrt(var + eps)) and the bound on the device's float32 result (module docstring)"""
    x = np.asarray(x, np.float64)
    inv = 1.0 / np.sqrt(np.asarray(var, np.float64) + eps)
    z = (x - mean) * inv
    tol = 1.01 * U32 * (inv * np.abs(mean) + 3.0 * np.abs(z)) + inv * dmean + 0.51 * np.abs(z) * dvar * inv * inv
    return np.clip(z, -clip, clip), tol + 1e-30


def _assert_normalised(got, x, mean, var, eps, clip, what, **kw):
    want, tol = _norm_ref(x, mean, var, eps, clip, **kw)
    err = np.abs(np.asarray(got, np.float64) - want)
    assert np.all(err <= tol), f"{what}: {float(np.max(err / tol)):.3g} x the bound"


def _sum_tol(vals, depth, total_after):
    """float64 sum on the device vs the reference sum, read as a difference of two running totals"""
    return (depth + REF_DEPTH) * U64 * float(np.abs(vals).sum()) + 2 * U64 * abs(total_after)


def _env(walker, n, seed=7, **cfg):
    from drloco_b200.vec_env import B200MimicVecEnv
    return B200MimicVecEnv(walker, num_envs=n, cfg=EnvConfig(env_id=walker, **cfg), seed=seed)


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _rms(mean, var, count):
    from oracle.env_oracle import RunningMeanStd
    r = RunningMeanStd(shape=np.shape(mean))
    r.mean, r.var, r.count = np.array(mean, np.float64), np.array(var, np.float64), count
    return r


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the epilogue parametrisation keeps the shapes where a fixed-order sum goes wrong
# ---------------------------------------------------------------------------------------------------------------------
def test_epilogue_cases_cover_the_ragged_grids():
    shapes = [(w,) + _launch_shape(w, n, b) for w, n, b in EPILOGUE_CASES]
    assert any(grid == 1 for _, _, _, grid, _, _, _ in shapes), "a single-block grid"
    assert any(last == 1 and ng > 1 for *_, ng, last in shapes), "a last group of one block"
    assert any(ng > 8 and ng % 8 for *_, ng, _ in shapes), "both loops of the final sum in one call"
    for G in (16, 32):
        assert any(g == G and pad > 0 for _, g, _, _, pad, _, _ in shapes), f"padding environments with G = {G}"
    assert any(grid > 2048 for _, _, _, grid, _, _, _ in shapes), "a grid above 2048 blocks"
    # the table of the shapes as documented
    assert [s[1:] for s in shapes] == [
        (16, 8, 1, 7, 1, 1), (16, 8, 17, 7, 2, 1), (16, 8, 513, 7, 33, 1), (16, 6, 683, 2, 43, 11),
        (16, 2, 32768, 1, 2048, 16), (16, 8, 8192, 0, 512, 16), (32, 3, 334, 1, 21, 14), (32, 4, 4096, 1, 256, 16)]


# ---------------------------------------------------------------------------------------------------------------------
# 1. statistics epilogue of the step kernel at production and ragged grids
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("walker,n,block", EPILOGUE_CASES, ids=[f"{w[:4]}-{n}-{b}" for w, n, b in EPILOGUE_CASES])
def test_step_statistics_epilogue_against_float64(walker, n, block):
    """Real physics, a few steps, some walkers dropped below the fall height (the last env among them: its warp-mate
    may be a padding environment).  Every step: the VecNormalize statistics against RunningMeanStd (SB3 1.0, two-pass
    np.var) fed the raw outputs, counts exactly; the normalised outputs to the float32 bound; every Monitor sum of
    ``env.stats()`` against the float64 sum of what the kernel exposes per environment."""
    from drloco_b200.vec_env import B200VecNormalize
    from oracle.env_oracle import RunningMeanStd
    env = _env(walker, n)
    env.debug_set(block_threads=block)
    G, epb, grid, pad, ngroups, _ = _launch_shape(walker, n, block)
    info = env.launch_info()
    assert (info["lanes_per_env"], info["block_threads"], info["grid_blocks"]) == (G, block, grid)
    depth = _epilogue_depth(epb, ngroups)
    vn = B200VecNormalize(env)
    D, A = env.obs_dim, env.act_dim
    eps, gamma = float(np.float32(vn.epsilon)), np.float32(vn.gamma)     # the kernels receive float32 parameters
    obs_rms, ret_rms = RunningMeanStd(shape=(D,)), RunningMeanStd(shape=())
    ob, rb = _RmsBound(depth, (D,)), _RmsBound(depth, ())
    vn.reset_tensor()
    ret_rms.update(np.zeros(n))                  # SB3 1.0 VecNormalize.reset
    rb.add(np.zeros(n))
    dyn_per_step = env.spec.frame_skip * 4       # RK4: four dynamics evaluations per substep
    rng = np.random.default_rng(n + block)
    n_done = 0
    for k in range(4):
        if k in (1, 3):                          # end some episodes: root below the fall height
            q, v, c = env.get_state()
            fall = rng.random(n) < 0.1
            fall[-1] = True
            q[fall, 2] = env.cfg.fall_z - 0.1
            env.set_state(q, v, c)
        ret_prev = vn.ret.cpu().numpy()
        st0 = env.stats()
        env.set_attr("ep_lens", [])
        act = torch.as_tensor(rng.uniform(-1, 1, (n, A)).astype(np.float32), device=env.device)
        nobs, nrew, done = vn.step_tensor(act)
        raw, rew = env.obs.cpu().numpy(), env.rew.cpu().numpy()
        d = done.cpu().numpy().astype(bool)
        ret_now = vn.ret.cpu().numpy()
        assert (ret_now[d] == 0).all()
        # the return the kernel's moments saw: ret*gamma + rew in float32; on a terminal step rew is +-0, so it is the
        # rounded product whether or not the compiler fused the two operations
        r = np.where(d, ret_prev * gamma, ret_now)
        rg = ret_prev.astype(np.float64) * gamma
        assert np.all(np.abs(r - (rg + rew)) <= 1.01 * U32 * (np.abs(rg) + np.abs(r)) + 1e-30)
        obs_rms.update(raw.astype(np.float64))
        ret_rms.update(r.astype(np.float64))
        ob.add(raw)
        rb.add(r)
        om, rm = vn.obs_rms, vn.ret_rms
        assert om.count == obs_rms.count and rm.count == ret_rms.count
        ob.check(om.mean, om.var, obs_rms, "obs_rms")
        rb.check(np.float64(rm.mean), np.float64(rm.var), ret_rms, "ret_rms")
        _assert_normalised(nobs.cpu().numpy(), raw, om.mean, om.var, eps, vn.clip_obs, "normalised obs")
        _assert_normalised(nrew.cpu().numpy(), rew, 0.0, rm.var, eps, vn.clip_reward, "normalised reward")
        # Monitor sums: this step's change against the float64 sums of the per-env values the kernel exposes
        st1 = env.stats()
        delta = {key: st1[key] - st0[key] for key in st1}
        nd = int(d.sum())
        n_done += nd
        assert delta["env_steps"] == n and delta["rew_steps"] == n           # padding environments do not count
        assert delta["episodes"] == nd and delta["falls"] + delta["timeouts"] + delta["blowups"] == nd
        assert delta["dyn_evals"] == n * dyn_per_step
        ex = env.extras().cpu().numpy().astype(np.float64)
        rec = env.episode_records()
        assert len(rec["ep_len"]) == nd
        ln, rt = rec["ep_len"], rec["ep_ret"]
        mr = (rt[ln > 1] / (ln[ln > 1] - 1).astype(np.float32)).astype(np.float32)
        for key, vals in (("pos_rew_sum", ex[:, 0]), ("vel_rew_sum", ex[:, 1]), ("com_rew_sum", ex[:, 2]),
                          ("abs_torque_sum", ex[:, 4]), ("moved_distance_sum", ex[d, 14]),
                          ("ep_len_sum", ln.astype(np.float64)), ("ep_ret_sum", rt.astype(np.float64)),
                          ("ep_mean_rew_sum", mr.astype(np.float64))):
            want = float(np.sum(vals))
            assert abs(delta[key] - want) <= _sum_tol(vals, depth, st1[key]), (key, delta[key], want)
    assert n_done >= 1
    vn.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. VecNormalize over a long horizon at 4096 envs against the float64 SB3 restatement
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_vecnormalize_long_horizon_against_sb3_float64():
    """W3D, 4096 envs, 300 steps of the numpy API with default settings, against SB3 1.0 VecNormalize restated in
    float64 (RunningMeanStd, ``ret`` in float64).

    The kernel keeps ``ret`` in float32 with gamma rounded to float32.  Per step the float32 return
    r32_k = fl32(g32 r32_{k-1} + rew) differs from r64_k = 0.99 r64_{k-1} + rew by e_k with
    |e_k| <= g32 |e_{k-1}| + |g32 - 0.99| |r64_{k-1}| + u32 (g32 |r32_{k-1}| + |r32_k|) (1 + u32) + 2 u64 (...),
    both reset to 0 together at the end of an episode.  That recursion is the asserted per-env bound b_k; at steady state
    it comes to (|g32 - 0.99| + 2 u32) / (1 - 0.99) ~ 1.4e-5 of the return.  The return statistics then differ by at
    most B = max_k mean_i b_k in the mean and by max_k mean_i (2 |r64| b + b^2) + 2 |mean| B + B^2 in the variance (the
    running statistics are weighted averages of E[x] and E[x^2] over every batch), on top of the one-pass bound."""
    from drloco_b200.vec_env import B200VecNormalize
    from oracle.env_oracle import RunningMeanStd
    n, steps = 4096, 300
    env = _env(W3D, n, seed=11)
    vn = B200VecNormalize(env)
    D, A = env.obs_dim, env.act_dim
    eps = float(np.float32(vn.epsilon))
    g32 = np.float32(vn.gamma)
    gd = abs(float(g32) - vn.gamma)
    _, epb, _, _, ngroups, _ = _launch_shape(W3D, n, env.launch_info()["block_threads"])
    depth = _epilogue_depth(epb, ngroups)
    obs_rms, ret_rms = RunningMeanStd(shape=(D,)), RunningMeanStd(shape=())
    ob, rb = _RmsBound(depth, (D,)), _RmsBound(depth, ())
    vn.reset()
    ret_rms.update(np.zeros(n))
    rb.add(np.zeros(n))
    ret64, r32, b = np.zeros(n), np.zeros(n, np.float32), np.zeros(n)
    drift_mean, drift_sq = 0.0, 0.0
    rng = np.random.default_rng(5)
    n_term = 0
    for k in range(steps):
        ret_prev = vn.ret.cpu().numpy()
        np.testing.assert_array_equal(ret_prev, r32)
        o, rw, d, infos = vn.step(rng.uniform(-1.5, 1.5, (n, A)).astype(np.float32))
        raw, rew = env.obs.cpu().numpy(), env.rew.cpu().numpy()
        ret_now = vn.ret.cpu().numpy()
        r = np.where(d, ret_prev * g32, ret_now)
        r64_prev = ret64
        ret64 = ret64 * vn.gamma + rew.astype(np.float64)
        b = g32 * b + gd * np.abs(r64_prev) + 1.0001 * U32 * (g32 * np.abs(ret_prev) + np.abs(r)) \
            + 2 * U64 * (np.abs(ret64) + np.abs(r64_prev))
        assert np.all(np.abs(r - ret64) <= b), float(np.max(np.abs(r - ret64) / b))
        drift_mean = max(drift_mean, float(b.mean()))
        drift_sq = max(drift_sq, float((2 * np.abs(ret64) * b + b * b).mean()))
        obs_rms.update(raw.astype(np.float64))
        ret_rms.update(ret64)
        ob.add(raw)
        rb.add(r)
        om, rm = vn.obs_rms, vn.ret_rms
        assert om.count == obs_rms.count and rm.count == ret_rms.count
        tm, tv = ob.check(om.mean, om.var, obs_rms, "obs_rms")
        # return statistics: the one-pass bound of the float32 returns plus their drift from the float64 ones
        rtol_m, rtol_v = rb.tols(ret_rms)
        rtol_m = float(rtol_m) + drift_mean
        rtol_v = float(rtol_v) + drift_sq + 2 * abs(ret_rms.mean) * drift_mean + drift_mean ** 2
        assert abs(rm.mean - ret_rms.mean) <= rtol_m and abs(rm.var - ret_rms.var) <= rtol_v, k
        _assert_normalised(o, raw, obs_rms.mean, obs_rms.var, eps, vn.clip_obs, "normalised obs", dmean=tm, dvar=tv)
        _assert_normalised(rw, rew, 0.0, ret_rms.var, eps, vn.clip_reward, "normalised reward", dvar=rtol_v)
        # terminal observations, normalised with the statistics just merged (SB3 VecNormalize.step_wait)
        idx = np.nonzero(d)[0]
        assert all("terminal_observation" not in infos[i] for i in np.nonzero(~d)[0][:64])
        if len(idx):
            got = np.stack([infos[i]["terminal_observation"] for i in idx])
            raw_t = env.terminal_obs.cpu().numpy()[idx]
            _assert_normalised(got, raw_t, obs_rms.mean, obs_rms.var, eps, vn.clip_obs, "terminal obs", dmean=tm,
                               dvar=tv)
            n_term += len(idx)
        ret64[d] = 0.0
        b[d] = 0.0
        r32 = np.where(d, np.float32(0), r).astype(np.float32)
    assert n_term > n                          # many episodes ended over the horizon
    vn.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. the VecNormalize kernels called directly on synthetic inputs
# ---------------------------------------------------------------------------------------------------------------------
def _lib():
    from drloco_b200 import lib
    return lib


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 29, 47, 64])
@pytest.mark.parametrize("n", [1, 7, 1000, 2 ** 16 + 3])
def test_moments_kernel_against_float64_sums(n, d):
    """vecnorm_moments_kernel: column sums and sums of squares, the count, and the return branch (ret <- ret*gamma +
    rew in place, its sums).  2^16 + 3 rows puts the grid at its 592-block cap, where every thread walks many rows and
    (d = 47) the strip stride (a multiple of d) leaves threads idle."""
    lib = _lib()
    L = lib.load()
    g = np.random.default_rng(n * 100 + d)
    obs = (g.standard_normal((n, d)) * 3 + g.uniform(-5, 5, d)).astype(np.float32)
    rew = g.uniform(-1, 2, n).astype(np.float32)
    ret0 = g.uniform(-20, 80, n).astype(np.float32)
    gamma = np.float32(0.99)
    dev = torch.device("cuda")
    t_obs, t_rew, t_ret = (torch.as_tensor(x, device=dev) for x in (obs, rew, ret0))
    packed = torch.full((2 * d + 3,), 7.0, dtype=torch.float64, device=dev)      # the call zeroes it
    depth = _moments_depth(n, d) + REF_DEPTH
    for with_rew in (False, True):
        lib.check(L.drl_vecnorm_moments(_ptr(t_obs), n, d, _ptr(t_rew) if with_rew else None,
                                        _ptr(t_ret) if with_rew else None, float(gamma), _ptr(packed), _stream()),
                  "drl_vecnorm_moments")
        p = packed.cpu().numpy()
        x = obs.astype(np.float64)
        assert p[2 * d] == n                                       # counted once, not once per block
        for got, vals in ((p[:d], x), (p[d:2 * d], x * x)):
            tol = depth * U64 * np.abs(vals).sum(axis=0)
            assert np.all(np.abs(got - vals.sum(axis=0)) <= tol)
        if not with_rew:
            assert p[2 * d + 1] == 0 and p[2 * d + 2] == 0
            np.testing.assert_array_equal(t_ret.cpu().numpy(), ret0)
            continue
        r = t_ret.cpu().numpy()
        rg = ret0.astype(np.float64) * gamma
        want = rg + rew
        assert np.all(np.abs(r - want) <= 1.01 * U32 * (np.abs(rg) + np.abs(want)))   # fused or two roundings
        r = r.astype(np.float64)
        for got, vals in ((p[2 * d + 1], r), (p[2 * d + 2], r * r)):
            assert abs(got - vals.sum()) <= depth * U64 * np.abs(vals).sum()


class _Comm:
    """a single-rank exchange (``drl_comm_create(1, 0, d)``) for the merge + normalisation kernel"""

    def __init__(self, d):
        self.L = _lib().load()
        self.h = C.c_void_p()
        _lib().check(self.L.drl_comm_create(1, 0, d, C.byref(self.h)), "drl_comm_create")

    def close(self):
        torch.cuda.synchronize()
        self.L.drl_comm_destroy(self.h)


def _moments(obs, rew, ret, gamma=0.99):
    n, d = obs.shape
    packed = torch.zeros(2 * d + 3, dtype=torch.float64, device=obs.device)
    _lib().check(_lib().load().drl_vecnorm_moments(_ptr(obs), n, d, _ptr(rew), _ptr(ret), float(gamma), _ptr(packed),
                                                   _stream()), "drl_vecnorm_moments")
    return packed


def _vn_step(comm, obs, rew, packed, rms_in, ret, done, clip_obs, clip_rew, eps, flags, sync_every):
    n, d = obs.shape
    obs_out, rms_out = torch.empty_like(obs), torch.empty_like(rms_in)
    rew_out = None if rew is None else torch.empty_like(rew)
    done_out = None if done is None else torch.empty_like(done)
    _lib().check(comm.L.drl_vecnorm_step(_ptr(obs), _ptr(obs_out), _ptr(rew), _ptr(rew_out), n, d, _ptr(packed),
                                         _ptr(rms_in), _ptr(rms_out), _ptr(ret), _ptr(done), _ptr(done_out),
                                         float(clip_obs), float(clip_rew), float(eps), flags, comm.h, sync_every,
                                         _stream()), "drl_vecnorm_step")
    return obs_out, rew_out, done_out, rms_out


def _chan(mean, var, count, bsum, bsumsq, bn):
    """csrc/vecnorm.cu::chan_merge in float64 (one-pass batch variance, clamped at 0)"""
    bm = bsum / bn
    bv = np.maximum(bsumsq / bn - bm * bm, 0.0)
    delta, tot = bm - mean, count + bn
    return mean + delta * bn / tot, (var * count + bv * bn + delta * delta * count * bn / tot) / tot, tot, \
        np.abs(bm) + np.abs(delta), bsumsq / bn + delta * delta


@pytest.mark.gpu
def test_vecnorm_step_kernel_flags_clipping_and_ill_conditioned_columns():
    """Every combination of the four flags (update obs statistics, norm_obs, norm_reward, update return statistics),
    clip bounds small enough that most values clip, values exactly at and next to +-clip, a constant column (var 0)
    and a column with |mean|/std = 1e3.  The merged statistics are checked against RunningMeanStd (two-pass np.var) to
    the one-pass bound of the module docstring: for the 1e3 column that is (11 c + 4) u64 (1 + 1e6) of the variance,
    about 1e-7 relative here, where the two-pass reference itself is exact to about 1e-14."""
    from oracle.env_oracle import RunningMeanStd
    n, d = 4099, 29
    g = np.random.default_rng(17)
    clip_obs, clip_rew = np.float32(0.5), np.float32(0.25)
    eps = float(np.float32(1e-8))
    obs = (g.standard_normal((n, d)) * 3 + g.uniform(-2, 2, d)).astype(np.float32)
    obs[:, 0] = 1.5                                                # constant column
    obs[:, 1] = (1000.0 + g.standard_normal(n)).astype(np.float32)  # |mean|/std = 1e3
    # column 2 with mean 0 and var + eps = 4 (inverse std 0.5 exactly): x = +-2 clip lands exactly on +-clip
    edge = np.array([2 * clip_obs, -2 * clip_obs, np.nextafter(2 * clip_obs, np.float32(9)),
                     np.nextafter(2 * clip_obs, np.float32(0)), -np.nextafter(2 * clip_obs, np.float32(0))], np.float32)
    obs[:len(edge), 2] = edge
    rew = (g.standard_normal(n) * 2).astype(np.float32)
    done = (g.random(n) < 0.3).astype(np.uint8)
    mean_in = g.uniform(-1, 1, d)
    var_in = g.uniform(0.5, 3, d)
    mean_in[0], var_in[0] = 1.5, 0.0
    mean_in[1], var_in[1] = 1000.0, 1.0
    mean_in[2], var_in[2] = 0.0, 4.0 - eps
    assert var_in[2] + eps == 4.0
    count_in, rmean_in, rvar_in, rcount_in = 37.0, 0.3, 1.7, 37.0
    rms_in = np.concatenate([mean_in, var_in, [count_in, rmean_in, rvar_in, rcount_in]])
    dev = torch.device("cuda")
    t_obs, t_rew, t_done = (torch.as_tensor(x, device=dev) for x in (obs, rew, done))
    t_rms = torch.as_tensor(rms_in, device=dev)
    ret0 = g.uniform(-5, 5, n).astype(np.float32)
    comm = _Comm(d)
    depth = _moments_depth(n, d)
    try:
        for flags in range(16):
            upd_obs, norm_obs, norm_rew, upd_ret = flags & 1, flags & 2, flags & 4, flags & 8
            t_ret = torch.as_tensor(ret0, device=dev)
            packed = _moments(t_obs, t_rew, t_ret)
            r = t_ret.cpu().numpy().astype(np.float64)                # ret*gamma + rew, as the moments kernel left it
            o, rw, dn, ro = _vn_step(comm, t_obs, t_rew, packed, t_rms, t_ret, t_done, clip_obs, clip_rew, eps, flags, 1)
            ro = ro.cpu().numpy()
            o, rw = o.cpu().numpy(), rw.cpu().numpy()
            np.testing.assert_array_equal(dn.cpu().numpy(), done)
            ret_after = t_ret.cpu().numpy()
            assert (ret_after[done == 1] == 0).all() and np.array_equal(ret_after[done == 0], r[done == 0].astype(np.float32))
            mean, var = ro[:d], ro[d:2 * d]
            if upd_obs:
                ref = _rms(mean_in, var_in, count_in)
                ref.update(obs.astype(np.float64))
                assert ro[2 * d] == ref.count
                bound = _RmsBound(depth, (d,))
                bound.sq = np.maximum(bound.sq, var_in + mean_in ** 2)
                bound.add(obs)
                bound.check(mean, var, ref, "obs statistics")
                assert var[0] == 0.0                                  # constant column: the one-pass variance is exact
            else:
                np.testing.assert_array_equal(ro[:2 * d + 1], rms_in[:2 * d + 1])
            if upd_ret:
                ref = _rms(rmean_in, rvar_in, rcount_in)
                ref.update(r)
                assert ro[2 * d + 3] == ref.count
                bound = _RmsBound(depth, ())
                bound.sq = max(float(bound.sq), rvar_in + rmean_in ** 2)
                bound.add(r)
                bound.check(np.float64(ro[2 * d + 1]), np.float64(ro[2 * d + 2]), ref, "return statistics")
            else:
                np.testing.assert_array_equal(ro[2 * d + 1:], rms_in[2 * d + 1:])
            if norm_obs:
                _assert_normalised(o, obs, mean, var, eps, float(clip_obs), f"obs, flags {flags}")
                assert (o[:, 0] == 0).all()
                assert np.mean(np.abs(o) == clip_obs) > 0.5                # most values clip
                if not upd_obs:
                    np.testing.assert_array_equal(o[:len(edge), 2], [clip_obs, -clip_obs, clip_obs,
                                                                     np.float32(clip_obs * np.float32(1 - 2 ** -24)),
                                                                     -np.float32(clip_obs * np.float32(1 - 2 ** -24))])
            else:
                np.testing.assert_array_equal(o, obs)
            if norm_rew:
                _assert_normalised(rw, rew, 0.0, ro[2 * d + 2], eps, float(clip_rew), f"reward, flags {flags}")
                assert np.mean(np.abs(rw) == clip_rew) > 0.5
            else:
                np.testing.assert_array_equal(rw, rew)
    finally:
        comm.close()


@pytest.mark.gpu
@pytest.mark.parametrize("K", [2, 3, 4])
def test_stats_sync_every_cycle_and_immediate_calls(K):
    """stats_sync_every = K against a float64 model of the documented semantics: the moments of cycle calls accumulate
    and merge on every K-th cycle call; the calls in between normalise with the statistics of the last merge (the
    statistics pass through bit for bit).  An immediate call (VecNormalize.reset) in the middle of a cycle merges its
    own moments at once and leaves the pending cycle alone.  The model is fed the moments the kernel was given and adds
    them in the same order, so only the Chan merge's rounding differs (the compiler may fuse its operations): at most a
    few u64 of each term it adds."""
    n, d = 1000, 29
    g = np.random.default_rng(K)
    eps = float(np.float32(1e-8))
    dev = torch.device("cuda")
    comm = _Comm(d)
    rms = np.concatenate([np.zeros(d), np.ones(d), [1e-4, 0.0, 1.0, 1e-4]])
    t_rms = torch.as_tensor(rms, device=dev)
    model = dict(mean=rms[:d].copy(), var=rms[d:2 * d].copy(), count=rms[2 * d], rmean=0.0, rvar=1.0, rcount=1e-4)
    pending, cyc = None, 0
    seq = ["cycle"] * (K + 1) + ["immediate"] + ["cycle"] * (2 * K)
    t_ret = torch.zeros(n, device=dev)
    n_merges = 0
    try:
        for j, kind in enumerate(seq):
            obs = (g.standard_normal((n, d)) * (1 + j) + j).astype(np.float32)
            t_obs = torch.as_tensor(obs, device=dev)
            if kind == "immediate":
                packed = _moments(t_obs, None, None)
                o, _, _, ro = _vn_step(comm, t_obs, None, packed, t_rms, None, None, 10.0, 10.0, eps, 1 | 2, 0)
                p = packed.cpu().numpy()
                merge, upd_ret = p, False
            else:
                rew = (g.standard_normal(n) + 0.5).astype(np.float32)
                done = (g.random(n) < 0.2).astype(np.uint8)
                t_rew, t_done = torch.as_tensor(rew, device=dev), torch.as_tensor(done, device=dev)
                packed = _moments(t_obs, t_rew, t_ret)
                o, rw, _, ro = _vn_step(comm, t_obs, t_rew, packed, t_rms, t_ret, t_done, 10.0, 10.0, eps, 15, K)
                p = packed.cpu().numpy()
                acc = p if cyc == 0 else pending + p
                if cyc + 1 >= K:
                    merge, pending, cyc = acc, None, 0
                else:
                    merge, pending, cyc = None, acc, cyc + 1
                upd_ret = True
            ro = ro.cpu().numpy()
            if merge is None:
                np.testing.assert_array_equal(ro, t_rms.cpu().numpy(), err_msg=f"call {j}: statistics of the last merge")
            else:
                n_merges += 1
                m, v, c, sm, sq = _chan(model["mean"], model["var"], model["count"], merge[:d], merge[d:2 * d],
                                        merge[2 * d])
                model.update(mean=m, var=v, count=c)
                assert ro[2 * d] == c, f"call {j} ({kind}): count {ro[2 * d]} vs {c}"
                assert np.all(np.abs(ro[:d] - m) <= 16 * U64 * (np.abs(m) + sm)), j
                assert np.all(np.abs(ro[d:2 * d] - v) <= 64 * U64 * (v + sq)), j
                if upd_ret:
                    m, v, c, sm, sq = _chan(model["rmean"], model["rvar"], model["rcount"], merge[2 * d + 1],
                                            merge[2 * d + 2], merge[2 * d])
                    model.update(rmean=m, rvar=v, rcount=c)
                    assert ro[2 * d + 3] == c and abs(ro[2 * d + 1] - m) <= 16 * U64 * (abs(m) + sm)
                    assert abs(ro[2 * d + 2] - v) <= 64 * U64 * (v + sq), j
                else:
                    np.testing.assert_array_equal(ro[2 * d + 1:], t_rms.cpu().numpy()[2 * d + 1:])
            _assert_normalised(o.cpu().numpy(), obs, ro[:d], ro[d:2 * d], eps, 10.0, f"obs of call {j}")
            if kind == "cycle":
                _assert_normalised(rw.cpu().numpy(), rew, 0.0, ro[2 * d + 2], eps, 10.0, f"reward of call {j}")
            t_rms = torch.as_tensor(ro, device=dev)
        assert n_merges == 1 + 1 + 2          # first cycle, the immediate call, the two cycles after it
    finally:
        comm.close()


def _check_terminal_records(words, done, tin, rms, d, eps, clip):
    cnt = int(words[:1].view(np.int32)[0])
    idx = np.nonzero(done)[0]
    assert cnt == len(idx)
    rec = words[4:4 + cnt * (d + 1)].reshape(cnt, d + 1)
    rows = rec[:, 0].copy().view(np.int32)
    assert np.array_equal(np.sort(rows), idx), "every finished row exactly once"
    _assert_normalised(rec[:, 1:], tin[rows], rms[:d], rms[d:2 * d], eps, clip, "terminal records")


@pytest.mark.gpu
def test_terminal_compaction_at_65536_rows():
    """vecnorm_terminal_compact_kernel at 65536 rows: the grid is capped at 592 blocks, so every warp walks many rows.
    All, some and no rows done; each finished row appears exactly once, normalised as the float64 reference says, and
    the header holds the count (twice in a row: the last block re-arms the counters)."""
    lib = _lib()
    L = lib.load()
    n, d = 65536, 29
    g = np.random.default_rng(9)
    eps = float(np.float32(1e-8))
    clip = 5.0
    dev = torch.device("cuda")
    tin = (g.standard_normal((n, d)) * 4).astype(np.float32)
    rms = np.concatenate([g.uniform(-1, 1, d), g.uniform(0.2, 3, d), [1e5, 0.0, 1.0, 1e5]])
    t_tin, t_rms = torch.as_tensor(tin, device=dev), torch.as_tensor(rms, device=dev)
    counters = torch.zeros(2, dtype=torch.int32, device=dev)
    out = torch.zeros(4 + n * (d + 1), device=dev)
    for name, done in (("all", np.ones(n, np.uint8)), ("some", (g.random(n) < 0.37).astype(np.uint8)),
                       ("none", np.zeros(n, np.uint8)), ("some again", (g.random(n) < 0.01).astype(np.uint8))):
        t_done = torch.as_tensor(done, device=dev)
        out.fill_(float("nan"))
        lib.check(L.drl_vecnorm_terminal_compact(_ptr(t_tin), _ptr(t_done), n, d, _ptr(t_rms), clip, eps, 1, _ptr(out),
                                                 _ptr(counters), _stream()), "drl_vecnorm_terminal_compact")
        _check_terminal_records(out.cpu().numpy(), done, tin, rms, d, eps, clip)
        assert counters.cpu().tolist() == [0, 0], name


@pytest.mark.gpu
@pytest.mark.parametrize("host_outputs", ["mapped", "copy"])
def test_vecnormalize_terminal_observations_every_env_done_at_65536(host_outputs):
    """Through B200VecNormalize at 65536 envs with every env finishing in the same step: "mapped" has the kernel write
    all records into pinned host memory; "copy" fetches the records past its fixed-size prefix with a second copy."""
    from drloco_b200.vec_env import B200VecNormalize
    n = 65536
    env = _env(W3D, n)
    env.debug_set(frame_skip_override=0)
    vn = B200VecNormalize(env)
    vn.host_outputs = host_outputs
    vn.reset()
    vn.step(np.zeros((n, env.act_dim), np.float32))
    q, v, c = env.get_state()
    q[:, 2] = env.cfg.fall_z - 0.1
    env.set_state(q, v, c)
    _, _, d, infos = vn.step(np.zeros((n, env.act_dim), np.float32))
    assert d.all()
    got = np.stack([infos[i]["terminal_observation"] for i in range(n)])
    om = vn.obs_rms
    _assert_normalised(got, env.terminal_obs.cpu().numpy(), om.mean, om.var, float(np.float32(vn.epsilon)),
                       vn.clip_obs, "terminal observations")
    vn.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. Monitor median past the staging capacity
# ---------------------------------------------------------------------------------------------------------------------
def _median_lengths(G):
    cap = MEDIAN_CAP[G]
    first = [1, 2, 703, 704, 705, 706, 1535, 1536, 1537, 1538, 2000, 3, 999, 1000, 17, 2000]
    assert {cap - 1, cap, cap + 1, cap + 2} <= set(first)
    return first


@pytest.mark.gpu
@pytest.mark.parametrize("walker", [W3D, W165])
def test_median_torque_past_the_staging_capacity(walker):
    """median_abs_torque_smoothed with episodes of chosen lengths (frozen physics; a fall is forced by putting the root
    below the fall height, the time-out is ep_dur_max = 2000): 1 and 2 steps, odd and even, both sides of the staging
    capacities of 704 (G = 16) and 1536 (G = 32) floats, where the radix select reads the rest of the history from
    global memory.  The two environments of a G = 16 warp get different lengths.  Actions give every actuator the same
    |a| from a small set (exact ties), runs of zero torque (key 0), and magnitudes a few float32 ulp apart (the last
    8-bit pass decides).  Reference: np.median of the float32 per-step torques since the env's reset, bit for bit for
    the first episode (numpy's float32 mean of the middle pair is 0.5f (lo + hi)); later episodes go through
    0.75 m + 0.25 prev in float32, within 1 ulp (the compiler may fuse it)."""
    n, ep_max = 16, 2000
    env = _env(walker, n, seed=3, ep_dur_max=ep_max, median_torque=True)
    env.debug_set(frame_skip_override=0)
    G = env.launch_info()["lanes_per_env"]
    assert G == LANES[walker]
    first = _median_lengths(G)
    if G == 16:
        assert all(first[2 * k] != first[2 * k + 1] for k in range(n // 2))
    plans = [[first[i]] + [first[(i + 5 + 3 * j) % n] for j in range(4)] for i in range(n)]
    pidx = np.zeros(n, int)
    env.reset()
    A = env.act_dim
    g = np.random.default_rng(1)
    base = np.float32(0.7)
    lowbits = [base]
    for _ in range(5):
        lowbits.append(np.nextafter(lowbits[-1], np.float32(2)))
    mags = np.array([0.25, 0.5, 1.0] + lowbits, np.float32)
    hist = [[] for _ in range(n)]
    prev = [None] * n
    ep = np.zeros(n, int)
    checked = {"first": 0, "later": 0, "long": 0}
    steps = ep_max + 700
    for k in range(steps):
        target = np.array([plans[i][pidx[i]] if pidx[i] < len(plans[i]) else ep_max for i in range(n)])
        fall = (ep + 1 == target) & (target < ep_max)
        if fall.any():
            q, v, c = env.get_state()
            q[fall, 2] = env.cfg.fall_z - 0.1
            env.set_state(q, v, c)
        m = g.choice(mags, n)
        m[(np.arange(n) + k // 41) % 4 == 0] = 0.0                        # runs of zero torque
        a = np.repeat(m[:, None], A, axis=1) * np.where(g.random((n, 1)) < 0.5, 1, -1).astype(np.float32)
        _, _, d, _ = env.step(a.astype(np.float32))
        tor = env.extras()[:, 4].cpu().numpy()
        for i in range(n):
            hist[i].append(tor[i])
        np.testing.assert_array_equal(d, fall | (ep + 1 == ep_max), err_msg=f"step {k}")
        if d.any():
            got = np.array(env.get_attr("median_abs_torque_smoothed"), np.float32)
            for i in np.nonzero(d)[0]:
                med = np.median(np.array(hist[i], np.float32))
                assert med.dtype == np.float32
                if prev[i] is None:
                    assert got[i] == med, (i, len(hist[i]), got[i], med)
                    checked["first"] += 1
                else:
                    want = np.float32(0.75) * med + np.float32(0.25) * prev[i]
                    assert abs(got[i] - want) <= np.spacing(want), (i, len(hist[i]), got[i], want)
                    checked["later"] += 1
                checked["long"] += len(hist[i]) > MEDIAN_CAP[G]
                prev[i], hist[i] = got[i], []
                pidx[i] += 1
        ep = np.where(d, 0, ep + 1)
    assert checked["first"] == n and checked["later"] >= n and checked["long"] >= 7


# ---------------------------------------------------------------------------------------------------------------------
# 5. episode ring wrap
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_episode_ring_wraps_oldest_first():
    """65536 envs (the ring's capacity) finish in one step, live four more steps and all finish in the fourth: 131072
    episodes, so the ring has wrapped once.  episode_records() returns exactly the second step's episodes (compared as a
    multiset of length, float32 return and RSI position); after set_attr('ep_lens', []) and one more such step, exactly
    that step's."""
    n = 65536
    env = _env(W3D, n)
    env.debug_set(frame_skip_override=0)
    env.reset()
    zeros = np.zeros((n, env.act_dim), np.float32)

    def fall_all():
        q, v, c = env.get_state()
        q[:, 2] = env.cfg.fall_z - 0.1
        env.set_state(q, v, c)

    def episode(length):
        """every env (just reset) lives `length` steps and finishes in the last one: (ep_len, ep_ret, rsi_pos)"""
        ep_ret = np.zeros(n, np.float32)
        rsi = None
        for j in range(length):
            if j == length - 1:
                fall_all()
            _, r, d, _ = env.step(zeros)
            ep_ret = ep_ret + r.astype(np.float32)                         # Monitor: float32 running sum
            assert d.all() if j == length - 1 else not d.any()
            if j == 0:
                rsi = env.get_state()[2][:, 1].copy()                      # cursor position after the first step
        return np.full(n, length), ep_ret, rsi

    def as_multiset(ln, rt, rp):
        a = np.stack([ln.astype(np.int64), rt.astype(np.float32).view(np.int32).astype(np.int64), rp.astype(np.int64)])
        return a[:, np.lexsort(a)]

    ln, rt, _ = episode(1)                     # ends the episodes begun at reset: the ring is full
    rec = env.episode_records()
    np.testing.assert_array_equal(rec["ep_len"], ln)
    np.testing.assert_array_equal(np.sort(rec["ep_ret"]), np.sort(rt))
    want = episode(4)                          # 131072 episodes: wrapped
    rec = env.episode_records()
    assert len(rec["ep_len"]) == n
    np.testing.assert_array_equal(as_multiset(rec["ep_len"], rec["ep_ret"], rec["rsi_pos"]), as_multiset(*want))
    env.set_attr("ep_lens", [])
    want = episode(2)
    rec = env.episode_records()
    assert len(rec["ep_len"]) == n
    np.testing.assert_array_equal(as_multiset(rec["ep_len"], rec["ep_ret"], rec["rsi_pos"]), as_multiset(*want))
    env.close()
