"""Ownership of the library's device buffers (csrc/dev_buf.h): every call that replaces a group of an env's buffers
(mocap tables, clip library, failure-weighted RSI table, speed profile, contact counters, debug dump) leaves the env
as a fresh env configured straight to the final values would be, and creating, configuring and destroying envs does
not leak device memory."""
import ctypes as C
import gc
from types import SimpleNamespace

import numpy as np
import pytest

from drloco_b200 import lib
from drloco_b200.config import EnvConfig
from drloco_b200.model import contact_body_mask
from drloco_b200.ref_trajecs import loco3d_trajecs as l3
from drloco_b200.ref_trajecs import straight_walk_trajecs as sw
from drloco_b200.vec_env import ADAPTIVE_RSI_BIN_STEPS
from drloco_b200.walkers import make_spec

pytestmark = pytest.mark.gpu

W3D, W165 = "StraightMimicWalker", "MimicWalker165cm65kg"
WEIGHTS = {W3D: ([0.5, 0.2, 0.3], [1.0, 1.0, 1.0]), W165: ([0.7, 0.3], [0.2, 0.8])}   # final, intermediate


@pytest.fixture(scope="module")
def clip_paths(tmp_path_factory):
    d = tmp_path_factory.mktemp("clips")
    paths = {W3D: [], W165: []}
    for k, n_steps in enumerate((3, 4, 2)):
        rows, lens = sw.synthetic_straight_rows(n_steps=n_steps, seed=20 + k)
        paths[W3D].append(str(d / f"s{k}.npz"))
        np.savez(paths[W3D][-1], rows=rows, step_len=lens)
    for k, seconds in enumerate((6.0, 9.0)):
        ang, vel = l3.synthetic_loco3d(duration_s=seconds, seed=30 + k)
        paths[W165].append(str(d / f"l{k}.npz"))
        np.savez(paths[W165][-1], angJoi=ang, angDJoi=vel)
    return paths


def _env(env_id, n, paths, **kw):
    from drloco_b200.vec_env import B200MimicVecEnv
    return B200MimicVecEnv(env_id, num_envs=n, cfg=EnvConfig(env_id=env_id, **kw), seed=11, mocap_path=paths,
                           clip_weights=WEIGHTS[env_id][0])


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _upload_mocap(env, spec):
    """drl_upload_mocap (and drl_set_mocap_clips for a library) of spec's tables, as the env's constructor does"""
    from drloco_b200.vec_env import B200MimicVecEnv
    B200MimicVecEnv._upload_mocap(SimpleNamespace(spec=spec, _lib=env._lib, _handle=env._handle))


def _set_clips(env, weights):
    t = env.spec.mocap
    first = np.ascontiguousarray(t.clip_first_step, np.int32)
    w = np.ascontiguousarray(weights, np.float64)
    lib.check(env._lib.drl_set_mocap_clips(env._handle, t.n_clips, _p(first), _p(w)), "drl_set_mocap_clips")


def _set_ars(env, lam, bin_samples):
    lib.check(env._lib.drl_set_adaptive_rsi(env._handle, lam, env.cfg.adaptive_rsi_halflife, bin_samples),
              "drl_set_adaptive_rsi")


def _set_speed_profile(env, speeds):
    buf = np.ascontiguousarray(speeds, np.float32)
    lib.check(env._lib.drl_set_speed_profile(env._handle, _p(buf) if buf.size else None, int(buf.size)),
              "drl_set_speed_profile")


def _set_contact_mask(env, mask):
    lib.check(env._lib.drl_set_contact_termination(env._handle, C.c_uint32(mask)), "drl_set_contact_termination")


def _contact_counts(env):
    import torch
    out = torch.zeros(env.num_envs, dtype=torch.int32, device=env.device)
    lib.check(env._lib.drl_get_contact_terminations(env._handle, C.c_void_p(out.data_ptr()), env._stream()),
              "drl_get_contact_terminations")
    return out.cpu().numpy()


def _run(env, acts):
    import torch
    outs = [env.reset_tensor().clone()]
    for a in acts:
        o, r, d = env.step_tensor(a)
        outs += [o.clone(), r.clone(), d.clone()]
    return dict(outs=torch.cat([x.float().flatten() for x in outs]).cpu().numpy(), stats=env.stats(),
                clips=env.clip_stats(), ars=env.adaptive_rsi_table(), contact=_contact_counts(env),
                cursor=env.get_state()[2])


@pytest.mark.parametrize("env_id", [W3D, W165])
def test_reconfiguration_equals_configuration(clip_paths, env_id):
    """env B walks every replacing call through an intermediate value to the final one; env A is configured straight
    to the final values.  From the same seed and actions both produce the same outputs, statistics, per-clip counts,
    failure-weighted RSI table and contact counts, bit for bit."""
    import torch
    n, steps = 512, 200
    paths = clip_paths[env_id]
    kw = dict(early_termination=True, ep_dur_max=60, adaptive_rsi=0.5, adaptive_rsi_halflife=50)
    a = _env(env_id, n, paths, contact_termination=True, **kw)
    b = _env(env_id, n, paths, **kw)
    final_w, other_w = WEIGHTS[env_id]
    bin_samples = ADAPTIVE_RSI_BIN_STEPS * b.spec.mocap.increment
    mask = contact_body_mask(b.spec.model)
    # the mocap calls refuse while failure-weighted RSI is on
    _set_ars(b, 0.0, bin_samples)
    _upload_mocap(b, make_spec(b.cfg, paths[1]))            # another recording
    _upload_mocap(b, b.spec)                                # the library with its final weights
    _set_clips(b, other_w)
    _set_clips(b, final_w)
    _set_ars(b, 0.5, bin_samples // 2)
    _set_ars(b, 0.0, bin_samples // 2)
    _set_ars(b, 0.5, bin_samples)
    _set_speed_profile(b, np.full(50, 1.1))
    _set_speed_profile(b, np.linspace(0.8, 1.2, 30))
    _set_speed_profile(b, [])
    _set_contact_mask(b, mask & -mask)                     # one of the listed bodies first
    _set_contact_mask(b, mask)
    b.debug_set(enable_dump=True)
    b.debug_set(enable_dump=False)
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    acts = torch.rand(steps, n, a.act_dim, device="cuda", generator=g) * 2 - 1
    ra, rb = _run(a, acts), _run(b, acts)
    a.close()
    b.close()
    np.testing.assert_array_equal(ra["outs"], rb["outs"])
    np.testing.assert_array_equal(ra["cursor"], rb["cursor"])
    np.testing.assert_array_equal(ra["contact"], rb["contact"])
    assert ra["stats"] == rb["stats"]
    for k in ra["clips"]:
        np.testing.assert_array_equal(ra["clips"][k], rb["clips"][k], err_msg=k)
    for k in ra["ars"]:
        np.testing.assert_array_equal(ra["ars"][k], rb["ars"][k], err_msg=k)
    # the run exercised what it compares
    assert ra["clips"]["episodes"].sum() > 0 and ra["ars"]["started"].sum() > 0 and ra["stats"]["episodes"] > 0


def test_lifecycle_does_not_leak(clip_paths):
    """create -> configure every replaceable group -> step -> destroy, ten times at 65536 envs.  A coarse check: the
    device is shared, so only losses above 64 MiB are caught.  Here state_f alone is 16 MiB and the debug dump 320 MiB,
    so losing either on every cycle fails it; the small tables are below its resolution."""
    import torch
    n = 65536
    paths = clip_paths[W3D]

    def cycle():
        env = _env(W3D, n, paths, integrator="euler", early_termination=True, adaptive_rsi=0.5,
                   contact_termination=True)                # the dump variant exists for Euler torque stepping only
        _set_speed_profile(env, np.full(40, 1.1))
        env.debug_set(enable_dump=True)
        env.reset_tensor()
        for _ in range(2):
            env.step_tensor(torch.zeros(n, env.act_dim, device="cuda"))
        torch.cuda.synchronize()
        env.close()

    def free():
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        return torch.cuda.mem_get_info()[0]

    cycle()                                                  # module load and caches
    free0 = free()
    for _ in range(10):
        cycle()
    assert free() >= free0 - (64 << 20)
