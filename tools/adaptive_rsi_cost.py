#!/usr/bin/env python
"""Step time with failure-weighted reference state initialisation off and on (EnvConfig.adaptive_rsi), in one process.

For each workload two environments are built, identical except for adaptive_rsi (0 / --lam), and stepped alternately
in blocks of --block steps (fixed, seeded actions; episodes end and reset as in training).  Each block is timed with
CUDA events around back-to-back drl_step calls: the fused step kernel, plus, with the option on, the one-block table
update kernel that drl_step enqueues after it.  --warmup untimed steps of both come first.  Prints one JSON line: per
workload the median block time per step off / on and their ratio, with the device name and power limit read in the
same process.  The option moves where episodes start, so the workload itself differs between the two: the episodes
per env-step of each variant are reported next to the times.  Runs on a GPU; there is no CPU path.

    python tools/adaptive_rsi_cost.py [--lam 0.5] [--blocks 8] [--block 50] [--out FILE]
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


def measure(env_id, integrator, n, blocks, block, warmup, lam, seed=11):
    envs = {w: B200MimicVecEnv(env_id, num_envs=n, seed=seed,
                               cfg=EnvConfig(env_id=env_id, integrator=integrator, adaptive_rsi=lam if w else 0.0))
            for w in (False, True)}
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    act_dim = envs[False].act_dim
    ring = torch.rand(64, n, act_dim, device="cuda", generator=g) * 2 - 1
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
    tab = envs[True].adaptive_rsi_table()
    ratio = tab["prob"] / tab["u"]
    for env in envs.values():
        env.close()
    off, on = float(np.median(times[False])), float(np.median(times[True]))
    return {"env_id": env_id, "integrator": integrator, "num_envs": n, "steps_per_variant": blocks * block,
            "adaptive_rsi": lam, "step_ms_off": off, "step_ms_on": on, "on_over_off": on / off,
            "block_ms_off": [round(x, 5) for x in times[False]], "block_ms_on": [round(x, 5) for x in times[True]],
            "episodes_off": stats[False]["episodes"], "episodes_on": stats[True]["episodes"],
            "episodes_per_env_step_off": stats[False]["episodes"] / stats[False]["env_steps"],
            "episodes_per_env_step_on": stats[True]["episodes"] / stats[True]["env_steps"],
            "n_bins": int(len(tab["u"])), "prob_over_u_min": float(ratio.min()), "prob_over_u_max": float(ratio.max())}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--blocks", type=int, default=8, help="timed blocks per variant (alternating)")
    ap.add_argument("--block", type=int, default=50, help="steps per timed block")
    ap.add_argument("--warmup", type=int, default=50, help="untimed steps of each variant first")
    ap.add_argument("--lam", type=float, default=0.5, help="EnvConfig.adaptive_rsi of the 'on' variant")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("adaptive_rsi_cost.py needs a CUDA device")
    res = {"tool": "adaptive_rsi_cost", **device_info(torch.cuda.current_device()),
           "method": "CUDA events around blocks of back-to-back drl_step calls (step kernel, plus the table update "
                     "kernel when on), median over blocks, adaptive_rsi off and on alternating in one process; "
                     "episodes per env-step over the warm-up and timed steps",
           "workloads": [measure(e, i, n, args.blocks, args.block, args.warmup, args.lam) for e, i, n in WORKLOADS]}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
