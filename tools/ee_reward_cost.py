#!/usr/bin/env python
"""Step-kernel time with the optional end-effector reward term off and on (EnvConfig.ee_weight), in one process.

For each workload two environments are built, identical except for ee_weight (0 and 0.3), and stepped alternately in
blocks of --block launches (fixed, seeded actions; episodes end and reset as in training).  Each block is timed with
CUDA events around back-to-back launches of the fused step kernel, after --warmup untimed launches of both.  Prints
one JSON line: per workload the median block time per launch off / on and their ratio, with the device name and
power limit read in the same process.  Runs on a GPU; there is no CPU path.

    python tools/ee_reward_cost.py [--blocks 8] [--block 50] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

from drloco_b200.config import EnvConfig  # noqa: E402
from drloco_b200.vec_env import B200MimicVecEnv  # noqa: E402

WORKLOADS = [("StraightMimicWalker", "rk4", 4096), ("MimicWalker165cm65kg", "rk4", 16384)]


def device_info(index):
    info = {"device": torch.cuda.get_device_name(index)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        pl, mx = [x.strip() for x in out.strip().split(",")]
        info.update(power_limit_w=float(pl), sm_max_mhz=int(mx))
    except (OSError, ValueError, subprocess.TimeoutExpired):
        info.update(power_limit_w=None, sm_max_mhz=None)
    return info


def measure(env_id, integrator, n, blocks, block, warmup, seed=11):
    envs = {w: B200MimicVecEnv(env_id, num_envs=n, seed=seed,
                               cfg=EnvConfig(env_id=env_id, integrator=integrator, ee_weight=w))
            for w in (0.0, 0.3)}
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    act_dim = envs[0.0].act_dim
    ring = torch.rand(64, n, act_dim, device="cuda", generator=g) * 2 - 1
    for env in envs.values():
        env.reset_tensor()
        for k in range(warmup):
            env.step_tensor(ring[k % 64])
    torch.cuda.synchronize()
    times = {w: [] for w in envs}
    k = 0
    for b in range(blocks):
        order = (0.0, 0.3) if b % 2 == 0 else (0.3, 0.0)          # alternate which variant runs first
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
    for env in envs.values():
        env.close()
    off, on = float(np.median(times[0.0])), float(np.median(times[0.3]))
    return {"env_id": env_id, "integrator": integrator, "num_envs": n, "launches_per_variant": blocks * block,
            "kernel_ms_off": off, "kernel_ms_on": on, "on_over_off": on / off,
            "block_ms_off": [round(x, 5) for x in times[0.0]], "block_ms_on": [round(x, 5) for x in times[0.3]],
            "episodes_off": stats[0.0]["episodes"], "episodes_on": stats[0.3]["episodes"]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--blocks", type=int, default=8, help="timed blocks per variant (alternating)")
    ap.add_argument("--block", type=int, default=50, help="launches per timed block")
    ap.add_argument("--warmup", type=int, default=50, help="untimed launches of each variant first")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ee_reward_cost.py needs a CUDA device")
    res = {"tool": "ee_reward_cost", **device_info(torch.cuda.current_device()),
           "method": "CUDA events around blocks of back-to-back step-kernel launches, median over blocks, "
                     "term off (ee_weight 0) and on (ee_weight 0.3) alternating in one process",
           "workloads": [measure(e, i, n, args.blocks, args.block, args.warmup) for e, i, n in WORKLOADS]}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
