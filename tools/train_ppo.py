#!/usr/bin/env python
"""Train the straight walker with PPO on GPU rollouts (mirror of reference drloco/train.py:77-139, next-tier demo).

Usage: python tools/train_ppo.py --envs 4096 --steps 16000000 --out gpurun_out/ppo_curve.json
       python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29511 \
              tools/train_ppo.py --envs 512 --steps 16000000 --out gpurun_out/ppo_8gpu.json     (data parallel)
       python tools/train_ppo.py --cpu-oracle --envs 8 --steps 1000000 --reference-hypers --out ...   (the same learner
              on the CPU oracle stack: the comparison curve of BASELINE.json configs[4])
       python tools/train_ppo.py --actuation pd --kp 300 --kv 10 ...   (PD position servos instead of torque motors)
       python tools/train_ppo.py --contact-termination ...   (DeepMimic early termination on non-foot floor contact)
       python tools/train_ppo.py --adaptive-rsi 0.5 ...   (failure-weighted reference state initialisation)
       python tools/train_ppo.py --mocap A.npz B.mat --clip-weights 1 2 ...   (a mocap library: several recordings,
              per-clip episode counts logged with every row)
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from drloco_b200.ppo import PPO, PPOConfig, evaluate_walking  # noqa: E402
from drloco_b200.vec_env import vec_env  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=int(16e6))
    ap.add_argument("--batch", type=int, default=0, help="samples per update (default: 32 steps per env)")
    ap.add_argument("--minibatch", type=int, default=0)
    ap.add_argument("--out", default="gpurun_out/ppo_curve.json")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--monitor", default="", help="directory: attach the TrainingMonitor (evaluation, checkpoints, "
                                                  "scalars with the reference's tag names) and write there")
    ap.add_argument("--cpu-oracle", action="store_true",
                    help="drive the learner with the CPU oracle stack (oracle/env_oracle.py) instead of the GPU env")
    ap.add_argument("--reference-hypers", action="store_true",
                    help="the reference's rollout shape: 16384 samples per update, minibatch 2048 (hypers.py:78-79)")
    ap.add_argument("--no-eval", action="store_true")
    ap.add_argument("--actuation", choices=("torque", "pd"), default="torque",
                    help="torque: the action is the motor force (the reference); pd: position servos (EnvConfig.actuation)")
    ap.add_argument("--kp", type=float, nargs="+", help="servo stiffness: one value or one per actuator (--actuation pd)")
    ap.add_argument("--kv", type=float, nargs="+", help="servo damping, as --kp (default 0)")
    ap.add_argument("--contact-termination", action="store_true",
                    help="end an episode when a body other than the feet touches the floor "
                         "(EnvConfig.contact_termination)")
    ap.add_argument("--adaptive-rsi", type=float, default=0.0, metavar="LAMBDA",
                    help="share of random RSI draws weighted towards the mocap phases where episodes end early "
                         "(EnvConfig.adaptive_rsi; 0 = off)")
    ap.add_argument("--mocap", nargs="+", metavar="PATH",
                    help="reference motion file(s); several make a mocap library (default: the shipped recording)")
    ap.add_argument("--clip-weights", type=float, nargs="+", metavar="W",
                    help="RSI weight of every --mocap clip (default: proportional to the clips' sample counts)")
    ap.add_argument("--ref-obs", type=int, nargs="+", metavar="K", default=[],
                    help="append the reference pose K control steps ahead to the observation, one frame per K "
                         "(EnvConfig.ref_obs_offsets; at most 3, strictly increasing)")
    args = ap.parse_args()
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("WORLD_SIZE", "1"), ("LOCAL_RANK", "0")))
    if world > 1:
        torch.cuda.set_device(local)
        import datetime
        # a short collective timeout: a rank that falls out of step must fail the run quickly, not hold the GPUs
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local),
                                             timeout=datetime.timedelta(seconds=90))
    env_cfg = None
    if args.actuation == "pd" or args.contact_termination or args.adaptive_rsi > 0.0 or args.ref_obs:
        if args.cpu_oracle:
            ap.error("--actuation pd, --contact-termination, --adaptive-rsi and --ref-obs run on the GPU env only")
        from drloco_b200.config import EnvConfig
        pd = dict()
        if args.actuation == "pd":
            gain = lambda g: None if g is None else (g[0] if len(g) == 1 else tuple(g))   # noqa: E731
            pd = dict(actuation="pd", pd_kp=gain(args.kp), pd_kv=gain(args.kv))
        env_cfg = EnvConfig(env_id="StraightMimicWalker", seed=33 + args.seed + 100 * rank,
                            contact_termination=args.contact_termination, adaptive_rsi=args.adaptive_rsi,
                            ref_obs_offsets=tuple(args.ref_obs), **pd)
    library = args.mocap is not None and len(args.mocap) > 1
    if (args.mocap or args.clip_weights) and args.cpu_oracle:
        ap.error("--mocap and --clip-weights run on the GPU env only")
    if args.cpu_oracle:
        from tools.oracle_tensor_env import OracleTensorEnv
        env = OracleTensorEnv("StraightMimicWalker", args.envs, seed=33 + args.seed)
    else:
        env = vec_env("StraightMimicWalker", num_envs=args.envs, seed=33 + args.seed + 100 * rank, norm_rew=True,
                      device=f"cuda:{local}", env_id_offset=rank * args.envs, cfg=env_cfg,
                      mocap_path=args.mocap if library else (args.mocap or [None])[0], clip_weights=args.clip_weights)
    cfg = PPOConfig(total_steps=args.steps)
    if args.reference_hypers:
        cfg.batch_size, cfg.minibatch_size = 4096 * 4, 512 * 4
    else:
        # the reference collects 16384 samples per update with 8 envs (2048 steps each); with thousands of envs keep
        # rollouts long enough for GAE to see consequences: 32 control steps per env per update
        cfg.batch_size = args.batch or args.envs * 32
        cfg.minibatch_size = args.minibatch or max(2048, cfg.batch_size // 8)
    agent = PPO(env, cfg, seed=args.seed)

    def cb(a, row):
        if library:
            # per-clip episode counts of this rank since the start, by the clip each episode started in
            cs = env.venv.clip_stats()
            row = dict(row, clip_episodes=cs["episodes"].tolist(),
                       clip_mean_ep_len=[round(float(s) / max(int(e), 1), 2) for s, e in zip(cs["ep_len_sum"],
                                                                                               cs["episodes"])])
        if rank == 0:
            print(json.dumps({k: (round(v, 4) if isinstance(v, float) else v) for k, v in row.items()}), flush=True)

    mon = None
    if args.monitor:
        from drloco_b200.training_monitor import TrainingMonitor
        mon = TrainingMonitor(agent, env.venv.cfg, args.monitor.rstrip("/") + "/", verbose=1)
        mon.on_training_start()
        agent.step_callback = mon.on_step
    t0 = time.time()
    agent.learn(args.steps, log_every=5, callback=cb)
    if mon:
        mon.on_training_end()
        print("checkpoints kept:", mon.saved, " steps to convergence:", mon.steps_to_convergence, flush=True)
    if not args.cpu_oracle:
        torch.cuda.synchronize()
    wall = time.time() - t0
    chk = agent.parameter_checksum()
    if world > 1:
        allc = [torch.zeros_like(chk) for _ in range(world)]
        torch.distributed.all_gather(allc, chk)
        lockstep = all(torch.equal(c, allc[0]) for c in allc)
    else:
        lockstep = True
    ev = ev2 = None
    if rank == 0 and not args.no_eval and not args.cpu_oracle:
        ev = evaluate_walking(agent.policy, env)
        print("evaluation (deterministic policy, 20 deterministic inits):", json.dumps(ev), flush=True)
        ev2 = evaluate_walking(agent.policy, env, steady_state_counters=True)
        print("evaluation with the training-time desired-velocity counter (Q3):", json.dumps(ev2), flush=True)
    ars = None
    if args.adaptive_rsi > 0.0:
        t = env.venv.adaptive_rsi_table()
        ars = {k: t[k].tolist() for k in ("step", "first", "width", "u", "started", "difficult", "prob")}
    clips = None
    if library:
        cs = env.venv.clip_stats()
        # file names only: a curve records which recordings it used, not where they were on the machine
        clips = [dict(c, path=None if c["path"] is None else os.path.basename(c["path"]),
                      **{k: int(cs[k][i]) for k in cs}) for i, c in enumerate(env.venv.mocap_clips())]
    if rank == 0:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"envs_per_rank": args.envs, "world": world, "backend": "cpu-oracle" if args.cpu_oracle else "b200",
                       "total_steps": agent.num_timesteps, "wall_s": wall,
                       "env_steps_per_s_incl_learning": agent.num_timesteps / wall,
                       "replicas_bit_identical": lockstep,
                       "actuation": args.actuation, "pd_kp": args.kp, "pd_kv": args.kv,
                       "contact_termination": args.contact_termination, "adaptive_rsi": args.adaptive_rsi,
                       "ref_obs_offsets": args.ref_obs, "obs_dim": int(env.venv.obs_dim) if not args.cpu_oracle else None,
                       "config": {k: v for k, v in vars(cfg).items()}, "curve": agent.log, "evaluation": ev,
                       "evaluation_steady_state_counters": ev2, "adaptive_rsi_table_at_end": ars,
                       "mocap_clips_at_end": clips}, f, indent=1)
        print("done: %.1f s, %.2e env-steps/s incl. learning, replicas bit-identical: %s"
              % (wall, agent.num_timesteps / wall, lockstep))
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
