#!/usr/bin/env python
"""Step time without reference-pose observations against 1 and 3 frames (EnvConfig.ref_obs_offsets), in one process.

For each workload three environments are built, identical except for ref_obs_offsets: () (off), (10,) and (5, 10, 20).
Same seed and actions, so the physics and the episodes are the same in all three: only the frames and the wider
statistics row differ.  They are stepped in rotation in blocks of --block steps (fixed, seeded actions; episodes end
and reset as in training; the order rotates from block to block).  Each block is timed with CUDA events around
back-to-back drl_step calls, so the time is the step kernel's.  --warmup untimed steps of each come first.  Prints one
JSON line: per workload the median block time per step of each variant and the ratios to off, with the device name and
power limit read in the same process.  Runs on a GPU; there is no CPU path.

    python tools/ref_obs_cost.py [--blocks 9] [--block 50] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

from drloco_b200.config import EnvConfig  # noqa: E402
from drloco_b200.vec_env import B200MimicVecEnv  # noqa: E402
from tools.adaptive_rsi_cost import device_info  # noqa: E402

WORKLOADS = [("StraightMimicWalker", "rk4", 4096), ("MimicWalker165cm65kg", "rk4", 16384)]
VARIANTS = {"off": (), "1 frame": (10,), "3 frames": (5, 10, 20)}


def measure(env_id, integrator, n, blocks, block, warmup, seed=11):
    envs = {name: B200MimicVecEnv(env_id, num_envs=n, seed=seed,
                                  cfg=EnvConfig(env_id=env_id, integrator=integrator, ref_obs_offsets=offs))
            for name, offs in VARIANTS.items()}
    names = list(envs)
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    ring = torch.rand(64, n, envs["off"].act_dim, device="cuda", generator=g) * 2 - 1
    for env in envs.values():
        env.reset_tensor()
        for k in range(warmup):
            env.step_tensor(ring[k % 64])
    torch.cuda.synchronize()
    times = {w: [] for w in envs}
    k = 0
    for b in range(blocks):
        order = names[b % 3:] + names[:b % 3]                         # rotate which variant runs first
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
    dims = {w: envs[w].obs_dim for w in envs}
    for env in envs.values():
        env.close()
    med = {w: float(np.median(times[w])) for w in envs}
    return {"env_id": env_id, "integrator": integrator, "num_envs": n, "steps_per_variant": blocks * block,
            "offsets": {w: list(VARIANTS[w]) for w in envs}, "obs_dim": dims,
            "step_ms": med, "over_off": {w: med[w] / med["off"] for w in envs},
            "block_ms": {w: [round(x, 5) for x in times[w]] for w in envs},
            "episodes_per_env_step": {w: stats[w]["episodes"] / stats[w]["env_steps"] for w in envs}}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--blocks", type=int, default=9, help="timed blocks per variant (rotating)")
    ap.add_argument("--block", type=int, default=50, help="steps per timed block")
    ap.add_argument("--warmup", type=int, default=50, help="untimed steps of each variant first")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ref_obs_cost.py needs a CUDA device")
    res = {"tool": "ref_obs_cost", **device_info(torch.cuda.current_device()),
           "method": "CUDA events around blocks of back-to-back drl_step calls (the step kernel), median over blocks, "
                     "off / 1 frame / 3 frames rotating in one process; episodes per env-step over the warm-up and "
                     "timed steps",
           "workloads": [measure(e, i, n, args.blocks, args.block, args.warmup) for e, i, n in WORKLOADS]}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
