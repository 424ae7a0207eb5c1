#!/usr/bin/env python
"""Step-kernel time with torque motors and with PD position servos (EnvConfig.actuation), in one process.

For each workload two environments are built, identical except for the actuation ("torque", and "pd" with
kp = --kp, kv = --kv on every actuator), and stepped alternately in blocks of --block launches (fixed, seeded actions;
episodes end and reset as in training).  Each block is timed with CUDA events around back-to-back launches of the
fused step kernel, after --warmup untimed launches of both.  Prints one JSON line: per workload the median block time
per launch in torque / PD mode and their ratio, with the device name and power limit read in the same process.  Runs
on a GPU; there is no CPU path.

    python tools/pd_actuation_cost.py [--blocks 8] [--block 50] [--kp 200] [--kv 5] [--out FILE]
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


def measure(env_id, integrator, n, blocks, block, warmup, kp, kv, seed=11):
    cfgs = {"torque": EnvConfig(env_id=env_id, integrator=integrator),
            "pd": EnvConfig(env_id=env_id, integrator=integrator, actuation="pd", pd_kp=kp, pd_kv=kv)}
    envs = {w: B200MimicVecEnv(env_id, num_envs=n, seed=seed, cfg=c) for w, c in cfgs.items()}
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    act_dim = envs["torque"].act_dim
    ring = torch.rand(64, n, act_dim, device="cuda", generator=g) * 2 - 1
    for env in envs.values():
        env.reset_tensor()
        for k in range(warmup):
            env.step_tensor(ring[k % 64])
    torch.cuda.synchronize()
    times = {w: [] for w in envs}
    k = 0
    for b in range(blocks):
        order = ("torque", "pd") if b % 2 == 0 else ("pd", "torque")   # alternate which variant runs first
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
    tq, pd = float(np.median(times["torque"])), float(np.median(times["pd"]))
    return {"env_id": env_id, "integrator": integrator, "num_envs": n, "launches_per_variant": blocks * block,
            "kernel_ms_torque": tq, "kernel_ms_pd": pd, "pd_over_torque": pd / tq,
            "block_ms_torque": [round(x, 5) for x in times["torque"]], "block_ms_pd": [round(x, 5) for x in times["pd"]],
            "episodes_torque": stats["torque"]["episodes"], "episodes_pd": stats["pd"]["episodes"],
            "blowups_torque": stats["torque"]["blowups"], "blowups_pd": stats["pd"]["blowups"]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--blocks", type=int, default=8, help="timed blocks per variant (alternating)")
    ap.add_argument("--block", type=int, default=50, help="launches per timed block")
    ap.add_argument("--warmup", type=int, default=50, help="untimed launches of each variant first")
    ap.add_argument("--kp", type=float, default=200.0, help="servo stiffness of every actuator in PD mode")
    ap.add_argument("--kv", type=float, default=5.0, help="servo damping of every actuator in PD mode")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("pd_actuation_cost.py needs a CUDA device")
    res = {"tool": "pd_actuation_cost", **device_info(torch.cuda.current_device()),
           "method": "CUDA events around blocks of back-to-back step-kernel launches, median over blocks, "
                     "torque and PD actuation alternating in one process",
           "pd_kp": args.kp, "pd_kv": args.kv,
           "workloads": [measure(e, i, n, args.blocks, args.block, args.warmup, args.kp, args.kv)
                         for e, i, n in WORKLOADS]}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
