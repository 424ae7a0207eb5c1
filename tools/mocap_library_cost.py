#!/usr/bin/env python
"""Step time of a single recording against a 3-clip mocap library (make_spec(mocap_path=[...])), in one process.

For each workload two environments are built, identical except for the mocap: the walker's default recording alone,
and a library of that recording plus two synthetic clips of the same walker (straight walking: 30-step gaits from
sw.synthetic_straight_rows; loco3d: 40 s and 80 s recordings from l3.synthetic_loco3d), written to a temporary
directory.  They are stepped alternately in blocks of --block steps (fixed, seeded actions; episodes end and reset as in
training).  Each block is timed with CUDA events around back-to-back drl_step calls, so the time is the step kernel's.
--warmup untimed steps of both come first.  Prints one JSON line: per workload the median block time per step of each
variant and their ratio, with the device name and power limit read in the same process.  The library changes which
motions the episodes follow, so the workload itself differs a little: episodes per env-step are reported next to the
times.  Runs on a GPU; there is no CPU path.

    python tools/mocap_library_cost.py [--blocks 8] [--block 50] [--out FILE]
"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

from drloco_b200.config import EnvConfig  # noqa: E402
from drloco_b200.ref_trajecs import loco3d_trajecs as l3  # noqa: E402
from drloco_b200.ref_trajecs import straight_walk_trajecs as sw  # noqa: E402
from drloco_b200.vec_env import B200MimicVecEnv  # noqa: E402
from tools.adaptive_rsi_cost import device_info  # noqa: E402

WORKLOADS = [("StraightMimicWalker", "rk4", 4096), ("MimicWalker165cm65kg", "rk4", 16384)]


def library_paths(env_id, tmp):
    """[None (the default recording), clip, clip]"""
    paths = [None]
    for k in (1, 2):
        p = os.path.join(tmp, f"{env_id}_{k}.npz")
        if env_id == "StraightMimicWalker":
            rows, lens = sw.synthetic_straight_rows(n_steps=30, seed=100 + k)
            np.savez(p, rows=rows, step_len=lens)
        else:
            ang, vel = l3.synthetic_loco3d(duration_s=40.0 * k, seed=100 + k)
            np.savez(p, angJoi=ang, angDJoi=vel)
        paths.append(p)
    return paths


def measure(env_id, integrator, n, blocks, block, warmup, tmp, seed=11):
    cfg = EnvConfig(env_id=env_id, integrator=integrator)
    envs = {False: B200MimicVecEnv(env_id, num_envs=n, seed=seed, cfg=cfg),
            True: B200MimicVecEnv(env_id, num_envs=n, seed=seed, cfg=cfg, mocap_path=library_paths(env_id, tmp))}
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    ring = torch.rand(64, n, envs[False].act_dim, device="cuda", generator=g) * 2 - 1
    for env in envs.values():
        env.reset_tensor()
        for k in range(warmup):
            env.step_tensor(ring[k % 64])
    torch.cuda.synchronize()
    times = {w: [] for w in envs}
    k = 0
    for b in range(blocks):
        order = (False, True) if b % 2 == 0 else (True, False)          # alternate which variant runs first
        for w in order:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            for i in range(block):
                envs[w].step_tensor(ring[(k + i) % 64])
            ev[1].record()
            ev[1].synchronize()
            times[w].append(ev[0].elapsed_time(ev[1]) / block)
        k += block
    stats = {w: envs[w].stats() for w in envs}
    clips = envs[True].mocap_clips()
    cs = envs[True].clip_stats()
    for env in envs.values():
        env.close()
    one, lib3 = float(np.median(times[False])), float(np.median(times[True]))
    return {"env_id": env_id, "integrator": integrator, "num_envs": n, "steps_per_variant": blocks * block,
            "step_ms_one_clip": one, "step_ms_library": lib3, "library_over_one_clip": lib3 / one,
            "block_ms_one_clip": [round(x, 5) for x in times[False]],
            "block_ms_library": [round(x, 5) for x in times[True]],
            "episodes_per_env_step_one_clip": stats[False]["episodes"] / stats[False]["env_steps"],
            "episodes_per_env_step_library": stats[True]["episodes"] / stats[True]["env_steps"],
            "library_clips": [dict(c, path=None if c["path"] is None else os.path.basename(c["path"]),
                                   episodes=int(cs["episodes"][i])) for i, c in enumerate(clips)]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--blocks", type=int, default=8, help="timed blocks per variant (alternating)")
    ap.add_argument("--block", type=int, default=50, help="steps per timed block")
    ap.add_argument("--warmup", type=int, default=50, help="untimed steps of each variant first")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("mocap_library_cost.py needs a CUDA device")
    with tempfile.TemporaryDirectory() as tmp:
        res = {"tool": "mocap_library_cost", **device_info(torch.cuda.current_device()),
               "method": "CUDA events around blocks of back-to-back drl_step calls (the step kernel), median over "
                         "blocks, one clip and a 3-clip library alternating in one process; episodes per env-step "
                         "over the warm-up and timed steps",
               "workloads": [measure(e, i, n, args.blocks, args.block, args.warmup, tmp) for e, i, n in WORKLOADS]}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
