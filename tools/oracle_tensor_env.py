"""tools/oracle_tensor_env.py — the CPU oracle stack behind the tensor API the PPO learner consumes (developer tool for
the learning-curve comparison of BASELINE.json configs[4]; NOT product code: it executes oracle/).

OracleVecNormalize(OracleVecEnv(OracleMonitor(OracleMimicEnv))) = the reference's
VecNormalize(DummyVecEnv([Monitor(MimicWalker3dEnv())] * n)) (drloco/common/utils.py:97-134) restated in numpy over the
float64 physics restatement; here it hands out CPU torch tensors so that drloco_b200.ppo.PPO can be run on it unchanged.
"""
import os
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

from drloco_b200.config import EnvConfig              # noqa: E402
from drloco_b200.walkers import make_spec             # noqa: E402
from oracle.env_oracle import OracleVecEnv, OracleVecNormalize   # noqa: E402
from oracle.physics import OraclePhysics              # noqa: E402


class _Inner:
    def __init__(self, venv, spec):
        self._v, self.spec = venv, spec
        # the oracle restates the reference's observation: the base width, no reference-pose frames
        self.num_envs, self.obs_dim, self.act_dim = venv.num_envs, spec.base_obs_dim, spec.act_dim
        self.device = torch.device("cpu")
        self._reset_counts()

    def _reset_counts(self):
        self._base = [(len(m.ep_lens), sum(m.ep_lens), sum(m.returns)) for m in self._v.envs]
        self._moved, self._steps, self._pos, self._vel = 0.0, 0, 0.0, 0.0

    def stats(self):
        ep = sum(len(m.ep_lens) - b[0] for m, b in zip(self._v.envs, self._base))
        ln = sum(sum(m.ep_lens) - b[1] for m, b in zip(self._v.envs, self._base))
        rt = sum(sum(m.returns) - b[2] for m, b in zip(self._v.envs, self._base))
        return dict(episodes=float(ep), ep_len_sum=float(ln), ep_ret_sum=float(rt), moved_distance_sum=self._moved,
                    pos_rew_sum=self._pos, vel_rew_sum=self._vel, rew_steps=float(max(self._steps, 1)))

    def reset_stats(self):
        self._reset_counts()


class OracleTensorEnv:
    def __init__(self, env_id, num_envs, seed=0):
        import random
        random.seed(seed)
        np.random.seed(seed)
        spec = make_spec(EnvConfig(env_id=env_id))
        self._venv = OracleVecEnv(spec, num_envs, lambda: OraclePhysics(spec.model))
        self._vn = OracleVecNormalize(self._venv)
        self.venv = _Inner(self._venv, spec)
        self.device = torch.device("cpu")
        self._raw_rew = torch.zeros(num_envs)

    def reset_tensor(self):
        return torch.from_numpy(self._vn.reset().astype(np.float32))

    def step_tensor(self, actions):
        a = actions.detach().cpu().numpy().astype(np.float32)
        o, r, d, infos = self._vn.step(a)
        inner = self.venv
        for m, dn in zip(self._venv.envs, d):
            inner._pos += m.env.pos_rew
            inner._vel += m.env.vel_rew
            inner._steps += 1
            if dn:
                inner._moved += float(m.moved_distance)
        self._raw_rew = torch.from_numpy(np.array([m.rewards[-1] if m.rewards else 0.0 for m in self._venv.envs],
                                                  np.float32))
        return (torch.from_numpy(o.astype(np.float32)), torch.from_numpy(r.astype(np.float32)),
                torch.from_numpy(d.astype(np.uint8)))

    def get_original_reward(self):
        return self._raw_rew
