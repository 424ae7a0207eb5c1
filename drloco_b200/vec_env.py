"""B200MimicVecEnv: N DeepMimic walker environments on one B200 behind the SB3 ``VecEnv`` surface.

Replaces, as one unit, what reference ``drloco.common.utils.vec_env`` (utils.py:97-134) builds:
``VecNormalize(SubprocVecEnv([Monitor(MimicWalker3dEnv())] * n))``.  The host side here is plumbing only — PyTorch owns
device memory and streams, ctypes passes raw pointers to libdrloco_b200.so (include/drloco_b200.h); every environment
step is one fused CUDA kernel launch (csrc/mimic_step.cu).  There is no CPU fallback.

Two ways to step:
  * SB3-compatible numpy API: ``reset() -> obs``, ``step_async(actions)``, ``step_wait() -> (obs, rews, dones, infos)``
    with ``infos[i]["terminal_observation"]`` for finished episodes (host<->device copies every call);
  * tensor API: ``step_tensor(actions_cuda) -> (obs, rew, done)`` — everything stays in HBM, nothing synchronises.
"""
from __future__ import annotations

import ctypes as C
import os
from collections.abc import Sequence
from typing import Any, List, Optional, Tuple, Union

import numpy as np
import torch

from . import cabi, config as cfgm, lib
from .model import contact_body_mask
from .ref_trajecs.base_ref_trajecs import CURSOR_STEPWISE
from .walkers import WalkerSpec, make_spec, speed_profile


class Box:
    """Minimal stand-in for gym.spaces.Box (gym is optional at run time)."""

    def __init__(self, low, high, shape=None, dtype=np.float32):
        self.dtype = np.dtype(dtype)
        self.low = np.broadcast_to(np.asarray(low, self.dtype), shape if shape is not None else np.shape(low)).copy()
        self.high = np.broadcast_to(np.asarray(high, self.dtype), self.low.shape).copy()
        self.shape = self.low.shape

    def sample(self):
        lo = np.where(np.isfinite(self.low), self.low, -1.0)
        hi = np.where(np.isfinite(self.high), self.high, 1.0)
        return np.random.uniform(lo, hi).astype(self.dtype)

    def __repr__(self):
        return f"Box({self.low.min()}, {self.high.max()}, {self.shape}, {self.dtype})"


class LazyInfos(Sequence):
    """``infos`` of a step: behaves like the list of per-env dicts SB3's VecEnv returns, but only the finished
    environments own a dict up front (``{"terminal_observation": ...}``); any other entry is created (and remembered) the
    first time it is touched.  Nothing is shared between entries or between steps."""

    __slots__ = ("_n", "_d")

    def __init__(self, n: int, filled: Optional[dict] = None):
        self._n, self._d = n, filled if filled is not None else {}

    def __len__(self):
        return self._n

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(self._n))]
        i = int(i)
        if i < 0:
            i += self._n
        if not 0 <= i < self._n:
            raise IndexError(i)
        d = self._d.get(i)
        if d is None:
            d = self._d[i] = {}
        return d

    def __iter__(self):
        return (self[i] for i in range(self._n))

    def __eq__(self, other):
        return len(other) == self._n and all(a == b for a, b in zip(self, other))

    def __repr__(self):
        return f"LazyInfos(n={self._n}, filled={sorted(self._d)})"


class _TerminalRows:
    """device -> host path of the terminal observations: the rows of finished environments are compacted by
    csrc/vecnorm.cu::vecnorm_terminal_compact_kernel into records { env index, d floats } behind a 4-word header.

    Three modes.  own buffers (B200MimicVecEnv): records are compacted in device memory and a fixed-size prefix of the
    record buffer is copied to pinned host memory; the rest is fetched only when more environments finished than the
    prefix holds.  host_words only (B200VecNormalize, host_outputs="mapped"): the kernel writes the records straight
    into that pinned host buffer (mapped into the device's address space) - no copy at all.  dev_words + host_words
    (host_outputs="copy"): both are tails of a larger output pack whose head-plus-prefix the caller copies itself."""

    PREFIX = 256

    def __init__(self, n: int, d: int, device, host_words=None, dev_words=None):
        self.n, self.d, self.device = n, d, device
        self.words = self.words_for(n, d)
        self.npre = 4 + min(n, self.PREFIX) * (d + 1)
        self.counters = torch.zeros(2, dtype=torch.int32, device=device)
        self.direct = host_words is not None and dev_words is None
        self.own_copy = host_words is None
        if self.direct:
            self.dev = None
            self.set_host(host_words)
        elif dev_words is not None:
            self.dev = dev_words
            self.set_host(host_words)
        else:
            self.dev = torch.zeros(self.words, dtype=torch.float32, device=device)
            self.set_host(torch.zeros(self.words, dtype=torch.float32).pin_memory())

    @staticmethod
    def words_for(n, d):
        return 4 + n * (d + 1)

    def set_host(self, host_words):
        self.host = host_words
        self.host_np = self.host.numpy()
        self.host_i = self.host_np.view(np.int32)

    def enqueue(self, libh, tobs, done, rms, clip_obs, eps, norm_obs, stream_ptr):
        dst = self.host if self.direct else self.dev
        lib.check(libh.drl_vecnorm_terminal_compact(_ptr(tobs), _ptr(done), self.n, self.d, _ptr(rms), float(clip_obs),
                                                    float(eps), int(norm_obs), _ptr(dst), _ptr(self.counters),
                                                    stream_ptr), "drl_vecnorm_terminal_compact")
        if self.own_copy:
            self.host[:self.npre].copy_(self.dev[:self.npre], non_blocking=True)

    def collect(self, dtype) -> dict:
        """after the stream has been synchronised: {env index: {"terminal_observation": row}}"""
        cnt = int(self.host_i[0])
        if cnt == 0:
            return {}
        need = 4 + cnt * (self.d + 1)
        if not self.direct and need > self.npre:         # more finished environments than the prefix holds (rare)
            self.host[self.npre:need].copy_(self.dev[self.npre:need], non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
        rec = self.host_np[4:need].reshape(cnt, self.d + 1)
        idx = self.host_i[4:need].reshape(cnt, self.d + 1)[:, 0]
        rows = rec[:, 1:].astype(dtype)                  # one copy = fresh memory for all terminal observations
        return {int(i): {"terminal_observation": rows[k]} for k, i in enumerate(idx.tolist())}


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


CLIP_STAT_NAMES = ("episodes", "ep_len_sum", "falls", "timeouts", "blowups")   # drl_get_clip_stats columns
ADAPTIVE_RSI_BIN_STEPS = 20      # failure-weighted RSI: a bin spans this many control steps of reference motion


def adaptive_rsi_bins(step_len, bin_samples: int, clip_first_step=None, clip_weight=None) -> dict:
    """Bin layout of the failure-weighted RSI table (drl_set_adaptive_rsi): runs of at most bin_samples consecutive
    samples inside each mocap step, in step order.  Per bin: ``step``, ``first`` sample, ``width``, and ``u``, the
    probability of the bin under the reference's RSI draw (a uniform step, then a uniform sample in it).  Over a mocap
    library (``clip_first_step`` [n_clips + 1], normalised ``clip_weight`` [n_clips]) the base draw picks clip c with
    probability clip_weight[c] first: u = clip_weight[c] / steps of c * width / step length."""
    step_len = np.asarray(step_len, np.int64)
    if clip_first_step is not None and len(clip_first_step) > 2:
        cf = np.asarray(clip_first_step, np.int64)
        w = np.asarray(clip_weight, np.float64)
        w = w / np.add.accumulate(w)[-1]          # normalised again, in order, as drl_set_mocap_clips does
        per_step = np.repeat(w / np.diff(cf), np.diff(cf))
    else:
        per_step = np.full(step_len.size, 1.0 / step_len.size)
    steps, first, width = [], [], []
    for s, n in enumerate(step_len.tolist()):
        f = np.arange(0, n, bin_samples)
        steps.append(np.full(f.size, s))
        first.append(f)
        width.append(np.minimum(bin_samples, n - f))
    steps, first, width = (np.concatenate(x).astype(np.int32) for x in (steps, first, width))
    u = per_step[steps] * width.astype(np.float64) / step_len[steps].astype(np.float64)
    return dict(step=steps, first=first, width=width, u=u)


class B200MimicVecEnv:
    """Batched MimicEnv.  Same attribute / method names as SB3's VecEnv (SURVEY.md §8b)."""

    metadata = {"render.modes": []}

    def __init__(self, env_id: str = cfgm.STRAIGHT_WALKER, num_envs: int = 4096, device="cuda:0",
                 seed: int = 33, cfg: Optional[cfgm.EnvConfig] = None,
                 mocap_path: Union[None, str, Sequence[Optional[str]]] = None, env_id_offset: int = 0,
                 lanes_per_env: int = 0, spec: Optional[WalkerSpec] = None, clip_weights=None):
        self._lib = lib.load()                       # raises when the CUDA library is missing
        if not torch.cuda.is_available():
            raise lib.DrlError("drloco_b200 needs a CUDA device (there is no CPU path)")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise lib.DrlError(f"device must be a CUDA device, got {device}")
        self.cfg = cfg or (spec.cfg if spec is not None else cfgm.EnvConfig(env_id=env_id, seed=seed))
        # mocap_path: one recording or a library of them (make_spec), clip_weights: the library's RSI clip weights
        self.spec = spec or make_spec(self.cfg, mocap_path, clip_weights)
        self.num_envs = int(num_envs)
        self.obs_dim, self.act_dim = self.spec.obs_dim, self.spec.act_dim
        m = self.spec.model
        self.observation_space = Box(-np.inf, np.inf, (self.obs_dim,), np.float64)
        self.action_space = Box(m.act_ctrlrange[:, 0], m.act_ctrlrange[:, 1], dtype=np.float32)   # mimic_env.py:256-262
        self._handle = C.c_void_p()
        c = self._make_config(seed, env_id_offset, lanes_per_env)
        lib.check(self._lib.drl_create(C.byref(c), C.byref(self._handle)), "drl_create")
        self._cm = cabi.pack_model(m)
        lib.check(self._lib.drl_upload_model(self._handle, C.byref(self._cm)), "drl_upload_model")
        if self.cfg.actuation == "pd":
            # position servos (EnvConfig.actuation): the action picks each servo's target in its joint's range, so
            # the policy acts in [-1, 1] (SB3 clips its samples to the action space before stepping)
            kp, kv = self.cfg.pd_gains(m.nu)
            lib.check(self._lib.drl_set_actuation(self._handle, cabi.ACTUATION_PD, kp.ctypes.data_as(C.c_void_p),
                                                  kv.ctypes.data_as(C.c_void_p)), "drl_set_actuation")
            self.action_space = Box(-1.0, 1.0, (m.nu,), dtype=np.float32)
        if self.cfg.contact_termination:
            # DeepMimic contact termination (EnvConfig.contact_termination): every body without a foot-corner site
            lib.check(self._lib.drl_set_contact_termination(self._handle, contact_body_mask(m)),
                      "drl_set_contact_termination")
        self._upload_mocap()
        offs = self.cfg.ref_obs_offsets
        if offs:
            # reference-pose observations (EnvConfig.ref_obs_offsets): every row gets one frame per offset
            self.spec.ref_frame_mirror()           # raises when the mirror table does not keep the qpos block
            arr = np.ascontiguousarray(offs, np.int32)
            lib.check(self._lib.drl_set_ref_obs(self._handle, len(offs), arr.ctypes.data_as(C.c_void_p)),
                      "drl_set_ref_obs")
        self._ars_bins = None
        if self.cfg.adaptive_rsi > 0.0:
            # failure-weighted RSI (EnvConfig.adaptive_rsi): bins of 20 control steps of reference motion
            bin_samples = ADAPTIVE_RSI_BIN_STEPS * self.spec.mocap.increment
            t = self.spec.mocap
            self._ars_bins = adaptive_rsi_bins(t.step_len, bin_samples, t.clip_first_step, t.clip_weight)
            lib.check(self._lib.drl_set_adaptive_rsi(self._handle, float(self.cfg.adaptive_rsi),
                                                     int(self.cfg.adaptive_rsi_halflife), bin_samples),
                      "drl_set_adaptive_rsi")
        with torch.cuda.device(self.device):
            N, D = self.num_envs, self.obs_dim
            dev = self.device
            # two output sets used alternately: a consumer working on step k (e.g. VecNormalize on a side stream)
            # is never overwritten by step k+1
            self._outs = [dict(obs=torch.zeros(N, D, device=dev), rew=torch.zeros(N, device=dev),
                               done=torch.zeros(N, dtype=torch.uint8, device=dev),
                               terminal_obs=torch.zeros(N, D, device=dev)) for _ in range(2)]
            self._cur = 0
            self._actions = torch.zeros(N, self.act_dim, device=dev)
            self._extras = torch.zeros(N, cabi.EXTRA_COUNT, device=dev)
            self._stats = torch.zeros(cabi.STATS_COUNT, dtype=torch.float64, device=dev)
            # pinned staging for the numpy API
            self._h_act = torch.zeros(N, self.act_dim).pin_memory()
            self._h_obs = torch.zeros(N, D).pin_memory()
            self._h_rew = torch.zeros(N).pin_memory()
            self._h_done = torch.zeros(N, dtype=torch.uint8).pin_memory()
            self._trows = _TerminalRows(N, D, dev)
        self._inj = None
        self._pending = False
        self._ep_lens_base = 0        # set_attr('ep_lens', []) marks the ring position (callback.py:69-70)
        self._closed = False
        self.launches = 0             # kernels launched through this env (bench: gpu_launches)
        self._config_epoch = 0        # bumped by every setter that changes what drl_step enqueues (captured graphs)

    # ------------------------------------------------------------------ construction helpers
    def _make_config(self, seed, env_id_offset, lanes_per_env) -> cabi.DrlConfig:
        s, cfg = self.spec, self.cfg
        c = cabi.DrlConfig()
        c.num_envs = self.num_envs
        c.device = self.device.index if self.device.index is not None else torch.cuda.current_device()
        c.frame_skip = s.frame_skip
        c.integrator = {"rk4": cabi.INTEGRATOR_RK4, "euler": cabi.INTEGRATOR_EULER}[cfg.integrator]
        c.ep_dur_max = cfg.ep_dur_max
        c.mirror_policy = 1 if s.mirror else 0
        c.phase_mode = cabi.PHASE_FROM_CURSOR if s.phase_from_cursor else cabi.PHASE_FROM_JOINTS
        c.n_phase_joints = len(s.phase_joints)
        for i, j in enumerate(s.phase_joints):
            c.phase_joints[i] = j
        c.eval_n_times = cfg.eval_n_times
        c.ctrl_freq = float(cfg.ctrl_freq)
        for i in range(4):
            c.rew_weights[i] = cfg.rew_weights[i]
        c.rew_scale, c.alive_bonus, c.fall_z = cfg.rew_scale, cfg.alive_bonus, cfg.fall_z
        c.seed, c.env_id_offset = int(seed) & (2 ** 64 - 1), int(env_id_offset)
        c.obs_dim, c.act_dim = s.base_obs_dim, s.act_dim      # the frames of ref_obs_offsets: drl_set_ref_obs
        oi, osn, ai, asn = s.mirror_tables()
        for i in range(s.base_obs_dim):
            c.mirror_obs_idx[i], c.mirror_obs_sign[i] = int(oi[i]), float(osn[i])
        for i in range(s.act_dim):
            c.mirror_act_idx[i], c.mirror_act_sign[i] = int(ai[i]), float(asn[i])
        c.lanes_per_env = lanes_per_env
        c.early_termination = int(bool(cfg.early_termination))
        hist_bytes = 4 * self.num_envs * max(1, cfg.ep_dur_max)
        self._median_torque = bool(getattr(cfg, "median_torque", False))
        if self._median_torque and hist_bytes > (4 << 30):
            raise lib.DrlError(f"median_torque: the torque history would need {hist_bytes >> 20} MiB")
        c.monitor_median_torque = int(self._median_torque)
        c.ee_weight, c.ee_scale = float(cfg.ee_weight), float(cfg.ee_scale)
        self._ee_term = c.ee_weight > 0.0
        return c

    def _upload_mocap(self):
        t = self.spec.mocap
        arrs = dict(ref=np.ascontiguousarray(t.ref, np.float64), off=np.ascontiguousarray(t.step_off, np.int32),
                    ln=np.ascontiguousarray(t.step_len, np.int32), left=np.ascontiguousarray(t.left_step, np.uint8),
                    vel=np.ascontiguousarray(t.step_vel, np.float64),
                    lastx=np.ascontiguousarray(t.step_last_comx, np.float64))
        pre = None if t.des_vel_prefix is None else np.ascontiguousarray(t.des_vel_prefix, np.float64)
        p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)   # noqa: E731
        lib.check(self._lib.drl_upload_mocap(self._handle, t.cursor_mode, t.increment, p(arrs["ref"]), t.n_samples,
                                             p(arrs["off"]), p(arrs["ln"]), p(arrs["left"]), p(arrs["vel"]),
                                             p(arrs["lastx"]), t.n_steps, t.com_z_col, p(pre), t.des_vel_window),
                  "drl_upload_mocap")
        if t.n_clips > 1:
            first = np.ascontiguousarray(t.clip_first_step, np.int32)
            w = np.ascontiguousarray(t.clip_weight, np.float64)
            lib.check(self._lib.drl_set_mocap_clips(self._handle, t.n_clips, p(first), p(w)), "drl_set_mocap_clips")

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # outputs of the most recent reset / step
    obs = property(lambda self: self._outs[self._cur]["obs"])
    rew = property(lambda self: self._outs[self._cur]["rew"])
    done = property(lambda self: self._outs[self._cur]["done"])
    terminal_obs = property(lambda self: self._outs[self._cur]["terminal_obs"])

    def _inject_tensors(self, inject):
        if inject is None:
            return None, None
        istep, pos = inject
        dev = self.device
        return (torch.as_tensor(np.asarray(istep, np.int32), device=dev), torch.as_tensor(np.asarray(pos, np.int32), device=dev))

    # ------------------------------------------------------------------ tensor API (no host synchronisation)
    def reset_tensor(self, mask: Optional[torch.Tensor] = None, inject=None) -> torch.Tensor:
        ii, ip = self._inject_tensors(inject)
        with torch.cuda.device(self.device):
            lib.check(self._lib.drl_reset(self._handle, _ptr(mask), _ptr(ii), _ptr(ip), _ptr(self.obs), self._stream()),
                      "drl_reset")
        self.launches += 1
        return self.obs

    def step_tensor(self, actions: torch.Tensor, inject=None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """actions: float32 CUDA tensor [N, act_dim].  Returns (obs, rew, done) device tensors owned by the env and
        overwritten two steps later (outputs alternate between two buffer sets); ``self.terminal_obs`` rows of done
        envs hold the pre-reset observation."""
        if actions.dtype != torch.float32 or not actions.is_cuda or not actions.is_contiguous() \
                or tuple(actions.shape) != (self.num_envs, self.act_dim):
            raise ValueError("actions must be a contiguous float32 CUDA tensor of shape [num_envs, act_dim]")
        ii, ip = self._inject_tensors(inject)
        self._cur ^= 1
        o = self._outs[self._cur]
        with torch.cuda.device(self.device):
            lib.check(self._lib.drl_step(self._handle, _ptr(actions), _ptr(o["obs"]), _ptr(o["rew"]), _ptr(o["done"]),
                                         _ptr(o["terminal_obs"]), _ptr(ii), _ptr(ip), self._stream()), "drl_step")
        self.launches += 2 if self._ars_bins is not None else 1    # + the failure-weighted RSI table update
        return o["obs"], o["rew"], o["done"]

    # ------------------------------------------------------------------ SB3 VecEnv API (numpy)
    def reset(self, inject=None) -> np.ndarray:
        self.reset_tensor(None, inject)
        self._h_obs.copy_(self.obs, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return self._h_obs.numpy().astype(np.float64)

    def step_async(self, actions, inject=None) -> None:
        a = np.ascontiguousarray(actions, np.float32).reshape(self.num_envs, self.act_dim)
        self._h_act.numpy()[...] = a
        self._actions.copy_(self._h_act, non_blocking=True)
        self.step_tensor(self._actions, inject)
        self._h_obs.copy_(self.obs, non_blocking=True)
        self._h_rew.copy_(self.rew, non_blocking=True)
        self._h_done.copy_(self.done, non_blocking=True)
        with torch.cuda.device(self.device):
            self._trows.enqueue(self._lib, self.terminal_obs, self.done, None, 0.0, 0.0, 0, self._stream())
        self.launches += 1
        self._pending = True

    def step_wait(self):
        if not self._pending:
            raise RuntimeError("step_wait() without step_async()")
        torch.cuda.current_stream(self.device).synchronize()
        self._pending = False
        obs = self._h_obs.numpy().astype(np.float64)
        rew = self._h_rew.numpy().astype(np.float64)
        done = self._h_done.numpy().astype(bool)
        infos = LazyInfos(self.num_envs, self._trows.collect(np.float64))
        return obs, rew, done, infos

    def step(self, actions, inject=None):
        self.step_async(actions, inject)
        return self.step_wait()

    def close(self) -> None:
        if not self._closed and self._handle:
            self._lib.drl_destroy(self._handle)
            self._handle = C.c_void_p()
            self._closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def seed(self, seed: Optional[int] = None):
        """``VecEnv.seed``: the reference calls ``env.seed(seed + rank * 100)`` when it builds its workers
        (utils.py:113).  Here it re-keys the counter-based RSI generator: env i then draws
        ``splitmix64(seed, env_id_offset + i, reset #)``.  Returns the per-env seeds as SB3 does."""
        if seed is None:
            return [None] * self.num_envs
        lib.check(self._lib.drl_set_seed(self._handle, C.c_uint64(int(seed) & (2 ** 64 - 1))), "drl_set_seed")
        return [int(seed) + i for i in range(self.num_envs)]

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False] * len(self._indices(indices))

    def get_images(self):
        raise NotImplementedError("rendering is out of scope (SURVEY.md §2 #15)")

    def _indices(self, indices) -> List[int]:
        if indices is None:
            return list(range(self.num_envs))
        if isinstance(indices, int):
            return [indices]
        return list(indices)

    # ---- attributes the reference's callback reads through get_attr (callback.py:106-108,142,162-164,227) ----
    def extras(self) -> torch.Tensor:
        with torch.cuda.device(self.device):
            lib.check(self._lib.drl_get_extras(self._handle, _ptr(self._extras), self._stream()), "drl_get_extras")
        self.launches += 1
        return self._extras

    def stats(self) -> dict:
        with torch.cuda.device(self.device):
            lib.check(self._lib.drl_get_stats(self._handle, _ptr(self._stats), self._stream()), "drl_get_stats")
        return dict(zip(cabi.STAT_NAMES, self._stats.cpu().tolist()))

    def stats_tensor(self) -> torch.Tensor:
        """packed float64 sums (all-reduce payload for multi-GPU episode statistics)."""
        with torch.cuda.device(self.device):
            lib.check(self._lib.drl_get_stats(self._handle, _ptr(self._stats), self._stream()), "drl_get_stats")
        return self._stats

    def reset_stats(self):
        lib.check(self._lib.drl_reset_stats(self._handle, self._stream()), "drl_reset_stats")

    def episode_records(self) -> dict:
        """the episodes finished since ``set_attr('ep_lens', [])`` (at most the ring capacity, oldest first): ``ep_len``,
        ``ep_ret`` and Monitor's position records ``rsi_pos``, ``et_pos``, ``difficult`` (monitor_wrapper.py:91-124)."""
        cap = 1 << 16
        dev = self.device
        with torch.cuda.device(dev):
            ln = torch.zeros(cap, dtype=torch.int32, device=dev)
            rt = torch.zeros(cap, dtype=torch.float32, device=dev)
            rp = torch.zeros(cap, dtype=torch.int32, device=dev)
            ep = torch.zeros(cap, dtype=torch.int32, device=dev)
            df = torch.zeros(cap, dtype=torch.uint8, device=dev)
            total = C.c_int64()
            lib.check(self._lib.drl_get_episode_ring(self._handle, _ptr(ln), _ptr(rt), cap, C.byref(total),
                                                     self._stream()), "drl_get_episode_ring")
            lib.check(self._lib.drl_get_episode_positions(self._handle, _ptr(rp), _ptr(ep), _ptr(df), cap,
                                                          self._stream()), "drl_get_episode_positions")
        total = total.value
        n_new = min(total - self._ep_lens_base, cap)
        idx = (np.arange(total - n_new, total) % cap) if n_new > 0 else np.zeros(0, np.int64)
        return dict(ep_len=ln.cpu().numpy()[idx], ep_ret=rt.cpu().numpy()[idx], rsi_pos=rp.cpu().numpy()[idx],
                    et_pos=ep.cpu().numpy()[idx], difficult=df.cpu().numpy()[idx].astype(bool))

    def episode_lengths(self) -> np.ndarray:
        return self.episode_records()["ep_len"]

    def get_attr(self, attr_name: str, indices=None) -> List[Any]:
        idx = self._indices(indices)
        if attr_name in cabi.EXTRA_NAMES:
            col = cabi.EXTRA_NAMES.index(attr_name)
            vals = self.extras()[:, col].cpu().numpy()
            return [float(vals[i]) for i in idx]
        if attr_name == "median_abs_torque_smoothed":      # monitor_wrapper.py:131
            if not self._median_torque:
                raise AttributeError("median_abs_torque_smoothed: the env was built with EnvConfig(median_torque=False)")
            with torch.cuda.device(self.device):
                out = torch.zeros(self.num_envs, device=self.device)
                lib.check(self._lib.drl_get_median_torque(self._handle, _ptr(out), self._stream()),
                          "drl_get_median_torque")
            vals = out.cpu().numpy()
            return [float(vals[i]) for i in idx]
        if attr_name in ("ee_rew", "mean_ep_ee_rew_smoothed"):   # the optional end-effector term (EnvConfig.ee_weight)
            if not self._ee_term:
                raise AttributeError(f"{attr_name}: the env was built with EnvConfig(ee_weight=0), the term is off")
            with torch.cuda.device(self.device):
                out = torch.zeros(self.num_envs, device=self.device)
                last, smoothed = (out, None) if attr_name == "ee_rew" else (None, out)
                lib.check(self._lib.drl_get_ee_reward(self._handle, _ptr(last), _ptr(smoothed), self._stream()),
                          "drl_get_ee_reward")
            vals = out.cpu().numpy()
            return [float(vals[i]) for i in idx]
        if attr_name == "contact_terminations":            # EnvConfig.contact_termination
            if not self.cfg.contact_termination:
                raise AttributeError("contact_terminations: the env was built with "
                                     "EnvConfig(contact_termination=False)")
            with torch.cuda.device(self.device):
                out = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
                lib.check(self._lib.drl_get_contact_terminations(self._handle, _ptr(out), self._stream()),
                          "drl_get_contact_terminations")
            vals = out.cpu().numpy()
            return [int(vals[i]) for i in idx]
        if attr_name == "ep_lens":
            # the reference returns one list per env and the callback flattens them (callback.py:227-230)
            lens = self.episode_lengths().tolist()
            return [lens] + [[] for _ in idx[1:]]
        if attr_name in ("et_positions", "difficult_rsi_phases", "rsi_positions"):
            # as ep_lens: one merged list (env 0).  rsi_positions = the finished episodes of the ring followed by the
            # entries of the episodes still running (Monitor appends on an episode's first step, monitor_wrapper.py:91-93)
            rec = self.episode_records()
            if attr_name == "et_positions":
                vals = rec["et_pos"].tolist()
            elif attr_name == "difficult_rsi_phases":
                vals = rec["rsi_pos"][rec["difficult"]].tolist()
            else:
                with torch.cuda.device(self.device):
                    run = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
                    lib.check(self._lib.drl_get_running_rsi_positions(self._handle, _ptr(run), self._stream()),
                              "drl_get_running_rsi_positions")
                run = run.cpu().numpy()
                vals = rec["rsi_pos"].tolist() + run[run >= 0].tolist()
            return [vals] + [[] for _ in idx[1:]]
        if attr_name in ("num_envs", "obs_dim", "act_dim"):
            return [getattr(self, attr_name)] * len(idx)
        if attr_name in ("ep_dur", "i_step", "pos"):
            cur = self.get_state()[2]
            col = {"i_step": 0, "pos": 1, "ep_dur": 3}[attr_name]
            return [int(cur[i, col]) for i in idx]
        raise AttributeError(f"B200MimicVecEnv has no per-env attribute {attr_name!r}")

    def set_attr(self, attr_name: str, value: Any, indices=None) -> None:
        if attr_name == "ep_lens":               # callback.py:69-70 empties the list roughly every 1M steps
            total = C.c_int64()
            lib.check(self._lib.drl_get_episode_ring(self._handle, None, None, 0, C.byref(total), self._stream()),
                      "drl_get_episode_ring")
            self._ep_lens_base = total.value
            return
        raise AttributeError(f"cannot set per-env attribute {attr_name!r}")

    def env_method(self, method_name: str, *args, indices=None, **kwargs) -> List[Any]:
        idx = self._indices(indices)
        self._config_epoch += 1
        if method_name == "activate_evaluation":             # mimic_env.py:245
            self._check_deterministic_inits("activate_evaluation")
            lib.check(self._lib.drl_set_eval_mode(self._handle, 1), "drl_set_eval_mode")
            return [None] * len(idx)
        if method_name == "activate_speed_control":          # mimic_env.py:298-327
            self.activate_speed_control(*args, **kwargs)
            return [None] * len(idx)
        if method_name == "get_walked_distance":              # mimic_env.py:295
            return self.get_attr("walked_distance", indices)
        if method_name == "get_COM_Z_position":               # mimic_env.py:128
            q = self.get_state()[0]
            return [float(q[i, 2]) for i in idx]
        raise AttributeError(f"env_method {method_name!r} is not served by the batched env")

    def activate_speed_control(self, speeds=(1.0, 1.0), speed_profile_duration: int = 10, plot_trajec=False):
        """MimicEnv.activate_speed_control (mimic_env.py:298-327) for every env of the batch: the desired-velocity
        observation follows the profile (indexed by the episode duration) and resets become deterministic.  The
        reference's own `_get_obs` then unpacks the scalar profile value with `*` and raises TypeError (run.py:76-79 is
        its only caller and is off by default, Q26); the evident intent - obs[des_vel] = profile value - is what runs
        here.  An empty ``speeds`` switches speed control off (not in the reference)."""
        self._config_epoch += 1
        if len(speeds):
            self._check_deterministic_inits("activate_speed_control")
        prof = speed_profile(speeds, speed_profile_duration, self.cfg.ctrl_freq) if len(speeds) else \
            np.zeros(0, np.float32)
        self.desired_walking_speed_trajectory = prof
        buf = np.ascontiguousarray(prof, np.float32)
        with torch.cuda.device(self.device):
            lib.check(self._lib.drl_set_speed_profile(self._handle, buf.ctypes.data_as(C.c_void_p) if buf.size else None,
                                                      int(buf.size)), "drl_set_speed_profile")

    def _check_deterministic_inits(self, who: str) -> None:
        """Deterministic inits start from the first eval_n_times steps of clip 0 (straight_walk_trajecs.py:237-265):
        over a walker3d library they must not run into the next clip."""
        t = self.spec.mocap
        n0 = int(t.clip_first_step[1])
        if t.n_clips > 1 and t.cursor_mode == CURSOR_STEPWISE and n0 < self.cfg.eval_n_times:
            raise ValueError(f"{who}: clip 0 of the mocap library has {n0} steps, fewer than "
                             f"eval_n_times = {self.cfg.eval_n_times}")

    def mocap_clips(self) -> List[dict]:
        """The clips of the mocap: per clip its ``path`` (None: the walker's default recording), ``first_step``,
        ``steps``, ``samples`` and normalised RSI ``weight``.  A single recording is one clip of weight 1."""
        t = self.spec.mocap
        out = []
        for k in range(t.n_clips):
            a, b = int(t.clip_first_step[k]), int(t.clip_first_step[k + 1])
            out.append(dict(path=self.spec.mocap_paths[k], first_step=a, steps=b - a,
                            samples=int(t.step_len[a:b].sum()), weight=float(t.clip_weight[k])))
        return out

    def clip_stats(self) -> dict:
        """Per-clip episode counts of a mocap library, by the clip each episode started in, since the env was built:
        int64 [n_clips] arrays ``episodes``, ``ep_len_sum``, ``falls`` (every terminal step that is neither a timeout
        nor a blow-up), ``timeouts`` and ``blowups``.  Exact, per env (per rank).  Raises with a single clip."""
        if self.spec.mocap.n_clips < 2:
            raise lib.DrlError("clip_stats: the env was built with a single mocap clip")
        with torch.cuda.device(self.device):
            out = torch.zeros(self.spec.mocap.n_clips, len(CLIP_STAT_NAMES), dtype=torch.int64, device=self.device)
            lib.check(self._lib.drl_get_clip_stats(self._handle, _ptr(out), self._stream()), "drl_get_clip_stats")
            out = out.cpu().numpy()
        return {name: out[:, k].copy() for k, name in enumerate(CLIP_STAT_NAMES)}

    def set_playback(self, on: bool = True) -> None:
        """kinematic playback mode (mimic_env.py:265-293): `step` skips the physics and sets qpos/qvel from the mocap
        after `refs.next()`; observation, reward, termination and Monitor logic run as usual."""
        self._config_epoch += 1
        lib.check(self._lib.drl_set_playback(self._handle, int(bool(on))), "drl_set_playback")

    def playback_ref_trajectories(self, timesteps: int = 2000):
        """MimicEnv.playback_ref_trajectories without the renderer: resets, then replays the mocap for ``timesteps``
        control steps and returns what a viewer would have shown plus the imitation reward of every step
        (``qpos [T,N,nq]``, ``qvel [T,N,nv]``, ``reward [T,N]``, ``done [T,N]``).  Unlike the reference it returns
        instead of closing the env and raising SystemExit (mimic_env.py:280-282)."""
        self.set_playback(True)
        try:
            self.reset()
            zeros = np.zeros((self.num_envs, self.act_dim), np.float32)
            Q, V, R, D = [], [], [], []
            for _ in range(timesteps):
                _, rew, done, _ = self.step(zeros)
                q, v, _ = self.get_state()
                Q.append(q); V.append(v); R.append(rew); D.append(done)
        finally:
            self.set_playback(False)
        return dict(qpos=np.stack(Q), qvel=np.stack(V), reward=np.stack(R), done=np.stack(D))

    # ------------------------------------------------------------------ state access (parity tests)
    def get_state(self):
        N = self.num_envs
        with torch.cuda.device(self.device):
            q = torch.zeros(N, self.spec.model.nv, device=self.device)
            v = torch.zeros_like(q)
            cur = torch.zeros(N, 4, dtype=torch.int32, device=self.device)
            lib.check(self._lib.drl_get_state(self._handle, _ptr(q), _ptr(v), _ptr(cur), self._stream()), "drl_get_state")
        self.launches += 1
        return q.cpu().numpy(), v.cpu().numpy(), cur.cpu().numpy()

    def set_state(self, qpos=None, qvel=None, cursor=None):
        dev = self.device
        q = None if qpos is None else torch.as_tensor(np.ascontiguousarray(qpos, np.float32), device=dev)
        v = None if qvel is None else torch.as_tensor(np.ascontiguousarray(qvel, np.float32), device=dev)
        c = None if cursor is None else torch.as_tensor(np.ascontiguousarray(cursor, np.int32), device=dev)
        with torch.cuda.device(dev):
            lib.check(self._lib.drl_set_state(self._handle, _ptr(q), _ptr(v), _ptr(c), self._stream()), "drl_set_state")
            torch.cuda.current_stream(dev).synchronize()
        self.launches += 1

    def set_det_init_counters(self, counts) -> None:
        """per-env `n_deterministic_inits` (straight_walk_trajecs.py:126): which mocap step each env's next deterministic
        init starts from; a batched evaluation passes arange(num_envs) % eval_n_times."""
        buf = np.ascontiguousarray(counts, np.int32).reshape(self.num_envs)
        with torch.cuda.device(self.device):
            lib.check(self._lib.drl_set_det_init_counters(self._handle, buf.ctypes.data_as(C.c_void_p)),
                      "drl_set_det_init_counters")

    def adaptive_rsi_table(self) -> dict:
        """The failure-weighted RSI table (EnvConfig.adaptive_rsi): per bin its mocap ``step``, ``first`` sample and
        ``width``, ``u`` (its probability under the reference's uniform draw), the decayed counts ``started`` and
        ``difficult``, ``prob`` (the probability of the current mixture) and, per env, ``env_bin``, the start bin of
        the running episode (-1: not counted).  Raises while the option is off."""
        if self._ars_bins is None:
            raise lib.DrlError("adaptive_rsi_table: the env was built with EnvConfig(adaptive_rsi=0)")
        nb = len(self._ars_bins["u"])
        with torch.cuda.device(self.device):
            t = torch.zeros(3, nb, dtype=torch.float64, device=self.device)
            eb = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
            lib.check(self._lib.drl_get_adaptive_rsi(self._handle, _ptr(t[0]), _ptr(t[1]), _ptr(t[2]), _ptr(eb),
                                                     self._stream()), "drl_get_adaptive_rsi")
            t, eb = t.cpu().numpy(), eb.cpu().numpy()
        return dict(self._ars_bins, started=t[0], difficult=t[1], prob=t[2], env_bin=eb)

    def set_adaptive_rsi_table(self, started, difficult) -> None:
        """Restore the counts of adaptive_rsi_table() (e.g. when resuming a run); the sampling tables are rebuilt at
        once.  float64 [n_bins] each, 0 <= difficult <= started.  Raises while the option is off."""
        if self._ars_bins is None:
            raise lib.DrlError("set_adaptive_rsi_table: the env was built with EnvConfig(adaptive_rsi=0)")
        nb = len(self._ars_bins["u"])
        s = np.ascontiguousarray(started, np.float64)
        f = np.ascontiguousarray(difficult, np.float64)
        if s.shape != (nb,) or f.shape != (nb,):
            raise ValueError(f"set_adaptive_rsi_table: started and difficult must have shape ({nb},)")
        with torch.cuda.device(self.device):
            lib.check(self._lib.drl_set_adaptive_rsi_counts(self._handle, s.ctypes.data_as(C.c_void_p),
                                                            f.ctypes.data_as(C.c_void_p)), "drl_set_adaptive_rsi_counts")

    def launch_info(self) -> dict:
        vals = [C.c_int32() for _ in range(4)]
        lib.check(self._lib.drl_launch_info(self._handle, *[C.byref(v) for v in vals]), "drl_launch_info")
        return dict(zip(("lanes_per_env", "block_threads", "grid_blocks", "smem_bytes"), [v.value for v in vals]))

    def debug_set(self, frame_skip_override=-1, block_threads=0, enable_dump=False):
        self._config_epoch += 1
        lib.check(self._lib.drl_debug_set(self._handle, frame_skip_override, block_threads, int(enable_dump)),
                  "drl_debug_set")

    def debug_read(self) -> np.ndarray:
        out = np.zeros((self.num_envs, 40, 32), np.float32)
        lib.check(self._lib.drl_debug_read(self._handle, out.ctypes.data_as(C.c_void_p), out.size), "drl_debug_read")
        return out


class RunningMeanStdView:
    """Read-only view with SB3's RunningMeanStd attribute names (mean, var, count)."""

    def __init__(self, mean, var, count):
        self.mean, self.var, self.count = mean, var, count


class B200VecNormalize:
    """SB3 VecNormalize semantics on the device (utils.py:130-132: norm_obs=True, norm_reward=norm_rew, clip 10/10,
    gamma=0.99, epsilon=1e-8), fused with the env: the step kernel itself keeps ``ret = ret*gamma + rew`` and leaves the
    batch moments of the observations it returns (csrc/mimic_step.cu epilogue, fixed-order sums: bit-reproducible), and
    ONE more kernel (csrc/vecnorm.cu::vecnorm_step_kernel) merges them into the running statistics and normalises.

    With ``torch.distributed`` initialised (one process per GPU of a node) the ranks' moments are exchanged inside that
    kernel through peer-mapped mailboxes over NVLink (``exchange="peer"``): no host-issued collective sits between the
    env step and the normalised observation.  ``exchange="nccl"`` keeps the all-reduce (ranks on different nodes, or
    no peer access).  Either way every rank holds bit-identical running statistics (SURVEY.md section 8e).

    ``stats_sync_every=K`` (opt-in, not SB3 semantics): exchange and merge the accumulated moments on every K-th step
    only; the steps in between are normalised with the statistics of the last merge.

    ``reset_update``: what ``reset()`` does to the statistics.  "sb3-1.0" (default) is SB3 1.0's ``VecNormalize.reset``:
    ``ret = 0`` and ``ret_rms.update(zeros)``, observation statistics untouched; "obs" also feeds the reset observations
    to ``obs_rms`` (later SB3 releases).  SB3 is not installed here: both are restated from memory (DESIGN.md section 4).
    """

    def __init__(self, venv: B200MimicVecEnv, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0,
                 clip_reward=10.0, gamma=0.99, epsilon=1e-8, distributed: Optional[bool] = None,
                 stats_sync_every: int = 1, exchange: str = "auto", reset_update: str = "sb3-1.0"):
        if reset_update not in ("sb3-1.0", "obs"):
            raise ValueError("reset_update must be 'sb3-1.0' or 'obs'")
        self.venv = venv
        self.num_envs, self.device = venv.num_envs, venv.device
        # the wrapper hands out float32 observations (what SB3 converts them to anyway); its space says so
        self.observation_space = Box(-np.inf, np.inf, (venv.obs_dim,), np.float32)
        self.action_space = venv.action_space
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon
        self.reset_update = reset_update
        D = venv.obs_dim
        self._D = D
        dev = self.device
        rms = torch.zeros(2 * D + 4, dtype=torch.float64, device=dev)
        rms[D:2 * D] = 1.0
        rms[2 * D] = 1e-4                      # RunningMeanStd(epsilon=1e-4)
        rms[2 * D + 2] = 1.0
        rms[2 * D + 3] = 1e-4
        self._rms = [rms, rms.clone()]
        self._cur = 0
        # batch moments of a step, written by the step kernel; one buffer per env output set
        self._packed = [torch.zeros(2 * D + 3, dtype=torch.float64, device=dev) for _ in range(2)]
        self._packed_reset = torch.zeros(2 * D + 3, dtype=torch.float64, device=dev)
        self.ret = torch.zeros(self.num_envs, device=dev)
        # normalised outputs of a step live side by side in one "pack" per buffer set - obs | rew | done | terminal
        # records - so that the numpy API fetches a whole step with ONE device-to-host copy
        N = self.num_envs
        self._w_obs, self._w_rew, self._w_done = N * D, N, (N + 3) // 4
        self._w_head = self._w_obs + self._w_rew + self._w_done
        self._pack = [torch.zeros(self._w_head + _TerminalRows.words_for(N, D), device=dev) for _ in range(2)]
        self._nobs = [p[:self._w_obs].view(N, D) for p in self._pack]
        self._nrew = [p[self._w_obs:self._w_obs + N] for p in self._pack]
        self._ndone = [p[self._w_obs + N:self._w_head].view(torch.uint8)[:N] for p in self._pack]
        self._k = 0
        # the normalisation kernel runs on a side stream so that it can overlap the next env step when the caller does
        # not consume the normalised tensors immediately
        with torch.cuda.device(dev):
            self._side = torch.cuda.Stream(device=dev)
            self._done_ev = [torch.cuda.Event(), torch.cuda.Event()]
        self._ev_used = [False, False]
        if distributed is None:
            distributed = torch.distributed.is_available() and torch.distributed.is_initialized() \
                and torch.distributed.get_world_size() > 1
        self.distributed = distributed
        self.stats_sync_every = max(1, int(stats_sync_every))
        self._lib = venv._lib
        self.launches = 0
        self._calls = 0                        # normalisation calls so far (host mirror of the device step counter)
        self._pending = None                   # exchange == "nccl" with stats_sync_every > 1: host-managed accumulation
        self._cycle = 0
        self._comm = C.c_void_p()
        self.exchange = self._setup_exchange(exchange)
        lib.check(self._lib.drl_attach_vecnorm(venv._handle, _ptr(self.ret), float(self.gamma),
                                               _ptr(self._packed[0])), "drl_attach_vecnorm")

    # -- statistics exchange ------------------------------------------------------------------------
    def _setup_exchange(self, mode: str) -> str:
        """"peer": mailboxes in every rank's HBM, mapped by the peers through CUDA IPC (one node, NVLink);
        "nccl": all-reduce of the packed moments; "local": single process."""
        dist = torch.distributed
        world = dist.get_world_size() if self.distributed else 1
        rank = dist.get_rank() if self.distributed else 0
        if mode not in ("auto", "peer", "nccl"):
            raise ValueError("exchange must be 'auto', 'peer' or 'nccl'")
        want_peer = world > 1 and mode in ("auto", "peer") and world <= 8
        with torch.cuda.device(self.device):
            if want_peer:
                comm = C.c_void_p()
                lib.check(self._lib.drl_comm_create(world, rank, self._D, C.byref(comm)), "drl_comm_create")
                handle = torch.zeros(64, dtype=torch.uint8)
                ok = self._lib.drl_comm_export(comm, C.c_void_p(handle.data_ptr())) == 0
                # every rank learns every handle (and whether every rank could export one)
                mine = torch.cat([handle, torch.tensor([1 if ok else 0], dtype=torch.uint8)]).to(self.device)
                allh = [torch.zeros_like(mine) for _ in range(world)]
                dist.all_gather(allh, mine)
                allh = torch.stack(allh).cpu()
                ok = bool(allh[:, 64].all())
                if ok:
                    table = allh[:, :64].contiguous()
                    ok = self._lib.drl_comm_connect(comm, C.c_void_p(table.data_ptr())) == 0
                flag = torch.tensor([1 if ok else 0], device=self.device)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                if int(flag.item()) == 1:
                    self._comm = comm
                    return "peer"
                self._lib.drl_comm_destroy(comm)
                if mode == "peer":
                    raise lib.DrlError("exchange='peer': CUDA IPC peer mapping is not available between these ranks")
            comm = C.c_void_p()
            lib.check(self._lib.drl_comm_create(1, 0, self._D, C.byref(comm)), "drl_comm_create")
            self._comm = comm
        return "nccl" if world > 1 else "local"

    # -- SB3 attribute surface ----------------------------------------------------------------------
    @property
    def obs_rms(self):
        self.synchronize()
        r, D = self._rms[self._cur], self._D
        return RunningMeanStdView(r[:D].cpu().numpy(), r[D:2 * D].cpu().numpy(), float(r[2 * D]))

    @property
    def ret_rms(self):
        self.synchronize()
        r, D = self._rms[self._cur], self._D
        return RunningMeanStdView(float(r[2 * D + 1]), float(r[2 * D + 2]), float(r[2 * D + 3]))

    norm_obs_buf = property(lambda self: self._nobs[self._k])
    norm_rew_buf = property(lambda self: self._nrew[self._k])

    def _attach_next(self):
        """the step about to be enqueued writes its moments into the buffer paired with the env's next output set"""
        lib.check(self._lib.drl_attach_vecnorm(self.venv._handle, _ptr(self.ret), float(self.gamma),
                                               _ptr(self._packed[self._k ^ 1])), "drl_attach_vecnorm")

    def _normalize(self, obs, rew, done, wait=True, packed=None, upd_obs=None, upd_ret=None, immediate=False,
                   out=None):
        """enqueue the exchange + merge + normalisation kernel for the env outputs just produced on the current stream.
        wait=True makes the current stream wait for the result (normal use); wait=False leaves it running on the side
        stream (``synchronize()`` / the next ``wait=True`` call / a stream sync picks it up)."""
        main = torch.cuda.current_stream(self.device)
        self._k ^= 1
        k = self._k
        # out: (obs, rew, done) destinations other than this buffer set's device pack - the numpy API passes pinned host
        # tensors, which the kernel then fills across PCIe itself
        nobs, nrew, ndone = out if out is not None else (self._nobs[k], self._nrew[k], self._ndone[k])
        if packed is None:
            packed = self._packed[k]
        upd_obs = self.training if upd_obs is None else upd_obs
        upd_ret = (self.training and rew is not None) if upd_ret is None else upd_ret
        K = self.stats_sync_every
        # wait=True: the kernel simply follows the env step on the caller's stream.  wait=False: it goes to the side
        # stream behind an event, so that the caller's next env step can overlap it.
        stream = main if wait else self._side
        if wait:
            if self._ev_used[k ^ 1]:                     # the previous call ran on the side stream: order after it
                main.wait_event(self._done_ev[k ^ 1])
        else:
            ready = torch.cuda.Event()
            ready.record(main)
        with torch.cuda.device(self.device), torch.cuda.stream(stream):
            if not wait:
                self._side.wait_event(ready)
            sync_every = 0 if immediate else K        # 0: exchange these moments now, outside the K-cycle (reset)
            if self.exchange == "nccl" and (upd_obs or upd_ret):
                # host-issued collective: the kernel then sees a single-rank exchange of already reduced moments
                sync_every = 0
                if K > 1 and not immediate:
                    if self._pending is None:
                        self._pending = torch.zeros_like(packed)
                    self._pending += packed
                    self._cycle += 1
                    if self._cycle >= K:
                        packed = self._pending.clone()
                        self._pending.zero_()
                        self._cycle = 0
                    else:
                        upd_obs = upd_ret = False
                if upd_obs or upd_ret:
                    if packed is self._packed[k] or packed is self._packed_reset:
                        packed = packed.clone()
                    torch.distributed.all_reduce(packed, op=torch.distributed.ReduceOp.SUM)
            flags = (1 if upd_obs else 0) | (2 if self.norm_obs else 0) | (4 if self.norm_reward else 0) | \
                (8 if upd_ret else 0)
            src, dst = self._rms[self._cur], self._rms[1 - self._cur]
            lib.check(self._lib.drl_vecnorm_step(_ptr(obs), _ptr(nobs), _ptr(rew), _ptr(nrew) if rew is not None else None,
                                                 self.num_envs, self._D, _ptr(packed), _ptr(src), _ptr(dst),
                                                 _ptr(self.ret), _ptr(done), _ptr(ndone),
                                                 float(self.clip_obs), float(self.clip_reward), float(self.epsilon),
                                                 flags, self._comm,
                                                 int(sync_every), C.c_void_p(stream.cuda_stream)), "drl_vecnorm_step")
            self.launches += 1
            self._calls += 1
            self._cur = 1 - self._cur
            if not wait:
                self._done_ev[k].record(self._side)
                self._ev_used[k] = True
            else:
                self._ev_used[k] = False

    def _guard_reuse(self):
        """before the env overwrites the output set it used two steps ago, make sure that step's normalisation is done."""
        k = self._k ^ 1
        if self._ev_used[k]:
            torch.cuda.current_stream(self.device).wait_event(self._done_ev[k])

    def synchronize(self):
        """make the current stream wait for the most recent normalisation."""
        if self._ev_used[self._k]:
            torch.cuda.current_stream(self.device).wait_event(self._done_ev[self._k])

    # -- tensor API -----------------------------------------------------------------------------------
    def reset_tensor(self, inject=None):
        self._guard_reuse()
        self.synchronize()
        obs = self.venv.reset_tensor(None, inject)
        self.ret.zero_()
        D = self._D
        if self.reset_update == "obs":
            # the reset observations update obs_rms (their moments come from the stand-alone moments kernel: the reset
            # launch has no statistics epilogue)
            pk = self._packed_reset
            with torch.cuda.device(self.device):
                lib.check(self._lib.drl_vecnorm_moments(_ptr(obs), self.num_envs, D, None, None, float(self.gamma),
                                                        _ptr(pk), self.venv._stream()), "drl_vecnorm_moments")
            self.launches += 1
            self._normalize(obs, None, None, packed=pk, upd_obs=self.training, upd_ret=False, immediate=True)
        else:
            # SB3 1.0 VecNormalize.reset: self.ret = zeros; if training: ret_rms.update(self.ret)
            pk = self._packed_reset
            pk.zero_()
            pk[2 * D] = float(self.num_envs)
            self._normalize(obs, None, None, packed=pk, upd_obs=False, upd_ret=self.training, immediate=True)
        return self.norm_obs_buf

    def step_tensor(self, actions, inject=None, wait=True):
        self._guard_reuse()
        self._attach_next()
        obs, rew, done = self.venv.step_tensor(actions, inject)
        self._normalize(obs, rew, done, wait)
        return self.norm_obs_buf, self.norm_rew_buf, done

    # -- SB3 numpy API -----------------------------------------------------------------------------------
    # float32 arrays are returned (SB3 converts observations to float32 tensors anyway).  Actions go through a pinned
    # staging buffer; obs / reward / done and a fixed-size prefix of the compacted terminal observations come back with
    # one asynchronous copy each and ONE stream synchronisation.  By default every returned array is a fresh copy.
    # `copy_outputs = False` hands out views of two alternating pinned buffers instead (valid until the second
    # following `step`; SB3's collect_rollouts reads `_last_obs` during the next step and stores it right after, which
    # that covers) and saves one 0.5 MB host copy per step.
    copy_outputs = True
    # "mapped": the kernels write the step's outputs straight into the pinned host pack (it is mapped into the device's
    # address space) - no D2H copy node.  "copy": they write the device pack and one copy moves obs | reward | done |
    # terminal-record prefix.  Set before the first numpy-API call.
    host_outputs = "mapped"

    def _host_buffers(self):
        if not hasattr(self, "_h"):
            assert self.host_outputs in ("mapped", "copy")
            N, D, A = self.num_envs, self._D, self.venv.act_dim
            # two alternating pinned host packs with the layout of the device packs
            hp = [torch.zeros(self._w_head + _TerminalRows.words_for(N, D)).pin_memory() for _ in range(2)]
            self._h = dict(act=torch.zeros(N, A).pin_memory(), pack=hp,
                           obs=[p[:self._w_obs].view(N, D) for p in hp],
                           rew=[p[self._w_obs:self._w_obs + N] for p in hp],
                           done=[p[self._w_obs + N:self._w_head].view(torch.uint8)[:N] for p in hp])
            self._h_np = dict(act=self._h["act"].numpy(), obs=[t.numpy() for t in self._h["obs"]],
                              rew=[t.numpy() for t in self._h["rew"]], done=[t.numpy() for t in self._h["done"]])
            self._hk = 0
            self._d_act = torch.zeros(N, A, device=self.device)
            if self.host_outputs == "mapped":
                self._trows = [_TerminalRows(N, D, self.device, host_words=p[self._w_head:]) for p in hp]
            else:
                # indexed by the DEVICE pack's parity; the host view is set when the step is collected
                self._trows = [_TerminalRows(N, D, self.device, host_words=hp[0][self._w_head:],
                                             dev_words=self._pack[k][self._w_head:]) for k in range(2)]
                self._n_copy = self._w_head + self._trows[0].npre
        return self._h

    def reset(self, inject=None):
        h = self._host_buffers()
        self._hk ^= 1
        nobs = self.reset_tensor(inject)
        h["obs"][self._hk].copy_(nobs, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        o = self._h_np["obs"][self._hk]
        return o.copy() if self.copy_outputs else o

    # The device side of a numpy-API step (H2D of the actions, env step, statistics kernel, terminal-row compaction and
    # the D2H copies) is captured into CUDA graphs, one per combination of the alternating buffer sets, and replayed
    # with a single launch.  `use_graph = False` (or an injected RSI draw, or the NCCL exchange) takes the eager path.
    use_graph = True

    def _enqueue_step(self, inject=None):
        h = self._h
        self._d_act.copy_(h["act"], non_blocking=True)
        self._guard_reuse()
        self._attach_next()
        obs, rew, done = self.venv.step_tensor(self._d_act, inject)
        self._hk ^= 1
        hk = self._hk
        mapped = self.host_outputs == "mapped"
        # exchange + merge + normalise; "mapped": results written straight into the pinned host pack
        self._normalize(obs, rew, done, True, out=(h["obs"][hk], h["rew"][hk], h["done"][hk]) if mapped else None)
        k = self._k
        tr = self._trows[hk if mapped else k]
        with torch.cuda.device(self.device):
            # terminal observations normalised with the statistics just merged (SB3 VecNormalize.step_wait), compacted
            # into the tail of the same pack
            tr.enqueue(self._lib, self.venv.terminal_obs, done, self._rms[self._cur], self.clip_obs, self.epsilon,
                       self.norm_obs, self.venv._stream())
        self.launches += 1
        if not mapped:
            # obs | rew | done | terminal-record prefix: one copy
            h["pack"][hk][:self._n_copy].copy_(self._pack[k][:self._n_copy], non_blocking=True)
        self._last = (tr, hk)

    def _graph_key(self):
        v = self.venv
        return (v._cur, self._k, self._cur, self._hk, bool(self.training), bool(self.norm_obs), bool(self.norm_reward),
                float(self.clip_obs), float(self.clip_reward), v._config_epoch, self.stats_sync_every)

    def step_async(self, actions, inject=None):
        self._host_buffers()
        self._h_np["act"][...] = np.asarray(actions, np.float32).reshape(self.num_envs, -1)
        if not self.use_graph or inject is not None or self.exchange == "nccl":
            return self._enqueue_step(inject)
        if not hasattr(self, "_graphs"):
            self._graphs, self._graph_warm = {}, 0
        if self._graph_warm < 2:                          # library one-time setup (function attributes) stays out of a capture
            self._graph_warm += 1
            return self._enqueue_step(None)
        key = self._graph_key()
        entry = self._graphs.get(key)
        v = self.venv
        if entry is None:
            # quiesce, then capture this step's enqueue sequence (it also executes nothing: replay right after)
            torch.cuda.synchronize(self.device)
            self._ev_used = [False, False]
            before = (v._cur, self._k, self._cur, self._hk, self._calls, v.launches, self.launches)
            g = torch.cuda.CUDAGraph()
            try:
                with torch.cuda.graph(g, stream=self._capture_stream()):
                    self._enqueue_step(None)
            except Exception:
                # capture is an optimisation: fall back to the eager path for good
                (v._cur, self._k, self._cur, self._hk, self._calls, v.launches, self.launches) = before
                self.use_graph = False
                torch.cuda.synchronize(self.device)
                return self._enqueue_step(None)
            after = (v._cur, self._k, self._cur, self._hk)
            dl = (v.launches - before[5], self.launches - before[6])
            (v._cur, self._k, self._cur, self._hk, self._calls, v.launches, self.launches) = before
            entry = self._graphs[key] = (g, after, dl)
        g, after, dl = entry
        g.replay()
        v._cur, self._k, self._cur, self._hk = after
        self._last = (self._trows[self._hk if self.host_outputs == "mapped" else self._k], self._hk)
        self._calls += 1
        v.launches += dl[0]
        self.launches += dl[1]
        self._ev_used = [False, False]

    def _capture_stream(self):
        if not hasattr(self, "_cap_stream"):
            with torch.cuda.device(self.device):
                self._cap_stream = torch.cuda.Stream(device=self.device)
        return self._cap_stream

    def step_wait(self):
        hn = self._h_np
        torch.cuda.current_stream(self.device).synchronize()
        tr, hk = self._last
        done = hn["done"][hk].astype(bool)
        if not tr.direct:
            tr.set_host(self._h["pack"][hk][self._w_head:])
        infos = LazyInfos(self.num_envs, tr.collect(np.float32))
        if self.copy_outputs:
            obs = self._h["obs"][hk].clone().numpy()                 # multi-threaded copy out of the pinned buffer
        else:
            obs = hn["obs"][hk]
        return obs, hn["rew"][hk].copy(), done, infos

    def step(self, actions, inject=None):
        self.step_async(actions, inject)
        return self.step_wait()

    def h2d_bytes_per_step(self) -> int:
        return self.num_envs * self.venv.act_dim * 4

    def d2h_bytes_per_step(self) -> int:
        """"mapped": bytes the kernels write into the pinned host pack per step: obs + reward + done + record header (+ one
        record of (D + 1) words per finished environment, not counted here); "copy": the size of the one copy"""
        if self.host_outputs == "copy":
            self._host_buffers()
            return self._n_copy * 4
        return self._w_head * 4 + 16

    def normalize_obs(self, obs: torch.Tensor) -> torch.Tensor:
        if not self.norm_obs:
            return obs
        r, D = self._rms[self._cur], self._D
        mean, var = r[:D].float(), r[D:2 * D]
        return torch.clamp((obs - mean) / torch.sqrt(var + self.epsilon).float(), -self.clip_obs, self.clip_obs)

    def get_original_obs(self):
        return self.venv.obs

    def get_original_reward(self):
        return self.venv.rew

    # -- save / load: same payload as the reference's pickled VecNormalize statistics (utils.py:183-184, 234-240) -----
    def state_dict(self) -> dict:
        self.synchronize()
        r, D = self._rms[self._cur].cpu().numpy(), self._D
        return dict(obs_mean=r[:D].copy(), obs_var=r[D:2 * D].copy(), obs_count=float(r[2 * D]),
                    ret_mean=float(r[2 * D + 1]), ret_var=float(r[2 * D + 2]), ret_count=float(r[2 * D + 3]),
                    clip_obs=self.clip_obs, clip_reward=self.clip_reward, gamma=self.gamma, epsilon=self.epsilon,
                    norm_obs=self.norm_obs, norm_reward=self.norm_reward)

    @staticmethod
    def _check_width(sd: dict, D: int) -> None:
        for k in ("obs_mean", "obs_var"):
            w = np.size(sd[k])
            if w != D:
                raise ValueError(f"VecNormalize statistics: {k} has {w} columns, the observation of this env has {D} "
                                 "(reference-pose frames change the width: EnvConfig.ref_obs_offsets)")

    def load_state_dict(self, sd: dict) -> None:
        D = self._D
        self._check_width(sd, D)
        r = np.zeros(2 * D + 4)
        r[:D], r[D:2 * D], r[2 * D] = sd["obs_mean"], sd["obs_var"], sd["obs_count"]
        r[2 * D + 1], r[2 * D + 2], r[2 * D + 3] = sd["ret_mean"], sd["ret_var"], sd["ret_count"]
        self._rms[self._cur].copy_(torch.as_tensor(r, device=self.device))
        for k in ("clip_obs", "clip_reward", "gamma", "epsilon", "norm_obs", "norm_reward"):
            setattr(self, k, sd[k])

    def save(self, path: str) -> None:
        import pickle
        with open(path, "wb") as f:
            pickle.dump(self.state_dict(), f)

    def save_sb3(self, path: str) -> None:
        """the same statistics as a pickle under SB3's class names (utils.py:183-184 writes such a file); see
        drloco_b200/checkpoint.py for what was and was not verified."""
        from .checkpoint import write_sb3_vecnormalize
        write_sb3_vecnormalize(path, {**self.state_dict(), "training": self.training}, self.num_envs)

    @staticmethod
    def load(path: str, venv: B200MimicVecEnv) -> "B200VecNormalize":
        """accepts this class's own file and a pickled SB3 ``VecNormalize`` (``envs/env_<ckpt>`` of the reference)."""
        import pickle
        sd = None
        try:
            with open(path, "rb") as f:
                sd = pickle.load(f)
        except (ImportError, AttributeError):        # SB3 / gym classes named by the pickle are not importable here
            pass
        if not isinstance(sd, dict):
            from .checkpoint import read_sb3_vecnormalize
            sd = read_sb3_vecnormalize(path)
        # before the wrapper attaches to the env: a refused file leaves the env as it was
        B200VecNormalize._check_width(sd, venv.obs_dim)
        vn = B200VecNormalize(venv)
        vn.load_state_dict(sd)
        if "training" in sd:                      # SB3's VecNormalize.load restores the pickled flag
            vn.training = bool(sd["training"])
        return vn

    # -- pass-through ----------------------------------------------------------------------------------------
    def get_attr(self, name, indices=None):
        return self.venv.get_attr(name, indices)

    def set_attr(self, name, value, indices=None):
        return self.venv.set_attr(name, value, indices)

    def env_method(self, name, *a, indices=None, **k):
        return self.venv.env_method(name, *a, indices=indices, **k)

    def seed(self, seed=None):
        return self.venv.seed(seed)

    def env_is_wrapped(self, wrapper_class, indices=None):
        return self.venv.env_is_wrapped(wrapper_class, indices)

    def close(self):
        if self._comm:
            torch.cuda.synchronize(self.device)
            self._lib.drl_attach_vecnorm(self.venv._handle, None, 0.0, None)
            self._lib.drl_comm_destroy(self._comm)
            self._comm = C.c_void_p()
        self.venv.close()


def vec_env(env_id: str, num_envs: int = 4, seed: int = 33, norm_rew: bool = True, load_path: Optional[str] = None,
            device="cuda:0", **kw) -> B200VecNormalize:
    """Drop-in for reference ``drloco.common.utils.vec_env`` (utils.py:97-134): same arguments, returns the normalised
    vectorised environment (here: B200VecNormalize(B200MimicVecEnv))."""
    venv = B200MimicVecEnv(env_id, num_envs=num_envs, device=device, seed=seed, **kw)
    if load_path is not None:
        return B200VecNormalize.load(load_path, venv)
    return B200VecNormalize(venv, norm_obs=True, norm_reward=norm_rew)
