#!/usr/bin/env python
"""bench.py — env-steps/s of the batched DeepMimic walker step (reward, termination and RSI resets included).

Contract (driver): ``python bench.py --gpus N --steps K --warmup W`` prints ONE JSON line on rank 0.
  * workload at N=1: BASELINE.json configs[1] — MimicWalker3d (StraightMimicWalker), straight-walking mocap, 4096 envs,
    random actions U(-1,1); for N>1 the same 4096 envs per GPU (weak scaling; envs are independent, the only exchange
    is the packed VecNormalize-moment all-reduce, SURVEY.md §8e).
  * ``value``: env-steps/s with actions already resident in HBM (tensor API: fused step kernel + VecNormalize kernels
    + the NCCL all-reduce when N>1), CUDA-event timed, max over ranks.
  * ``e2e``: the same metric through the SB3-facing numpy API (B200VecNormalize.step on HOST float32 actions; H2D of the
    actions and D2H of obs/reward/done inside the timed region).
  * ``roofline``: the step kernel is neither HBM- nor tensor-bound (SURVEY.md §8d): reported against HBM with the
    algorithmic 425 B/env-step, plus an ``fp32`` object against the FFMA peak measured in the same run.
  * ``cpu_baseline``: the oracle stack (reference env logic restated in numpy + float64 MuJoCo-restatement physics in C)
    on a bounded sample, single core ("port").
  * ``--impl reference``: the same oracle stack on all host cores, one process per core (what SubprocVecEnv does).
  * ``--dump-outputs DIR``: the outputs of the headline leg's last timed step as DIR/<name>.npy (see write_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

ENV_ID = "StraightMimicWalker"
W3D_WORKLOAD = ("MimicWalker3d straight walking, %d batched envs per GPU, random-action step+reward throughput "
                "(BASELINE.json configs[1])")
ENVS_PER_GPU = 4096
ALGO_BYTES_PER_ENV_STEP = 425.0        # SURVEY.md §8d / DESIGN.md
ALGO_FLOP_PER_EVAL = 16.0e3            # DESIGN.md §3: algorithmic flops of one dynamics evaluation (W3D)
W165 = "MimicWalker165cm65kg"


def algo_flop_per_env_step(env_id: str, integrator: str, frame_skip: int) -> float:
    """evaluations per control step (frame_skip x 4 RK4 stages, or x 1 for Euler) x flops per evaluation; the W165
    evaluation is scaled from W3D by (19/14)^2 (dense parts) as in DESIGN.md section 3."""
    per_eval = ALGO_FLOP_PER_EVAL * ((19 / 14) ** 2 if env_id == W165 else 1.0)
    return per_eval * frame_skip * (4 if integrator == "rk4" else 1)


def profiled_traffic(env_id: str, n: int, integrator: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of one step-kernel launch, from the committed ncu summary of the
    current kernel (profiles/step_kernel_traffic.json, written by tools/ncu_summary.py from the .ncu-rep); None when no
    capture exists for this shape."""
    path = os.path.join(REPO, "profiles", "step_kernel_traffic.json")
    try:
        with open(path) as f:
            table = json.load(f)
    except (OSError, ValueError):
        return None, None
    for row in table.get("captures", []):
        if row.get("env_id") == env_id and row.get("num_envs") == n and row.get("integrator") == integrator:
            return row.get("dram_bytes"), row.get("source")
    return None, None


def _peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region.  nvidia-smi takes up to a second to start on
    an 8-GPU box while a timed region lasts tens of milliseconds, so the sampler is started well before (`start`), every
    sample is stamped with the host clock, and only the samples between `begin()` and `end()` are reported."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "10"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        t0, t1 = self.t0 or 0.0, (self.t1 or time.time()) + 0.02       # a sample is printed up to one period late
        inside = [r for t, r in self.rows if t0 <= t <= t1]
        rows = inside if inside else [r for _, r in self.rows[-3:]]      # (region shorter than one period)
        sm = sorted(int(r[0]) for r in rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in rows if len(r) >= 6 for k in range(4) if r[2 + k].lower() == "active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "samples_inside_timed_regions": len(inside)}


def fp32_peak_tflops(device_index: int) -> float:
    """sustained FFMA rate measured by the library's own probe kernel (csrc/vecnorm.cu::ffma_probe_kernel)."""
    import ctypes as C

    from drloco_b200 import lib
    out = C.c_double()
    lib.check(lib.load().drl_fp32_peak_probe(device_index, C.byref(out)), "drl_fp32_peak_probe")
    return out.value


DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(directory: str, arrays: dict, shared: dict = None, limit: int = DUMP_LIMIT_BYTES) -> None:
    """DIR/<name>.npy for every per-environment output array (first axis = environment) and every ``shared`` array
    (written whole).  Above ``limit`` bytes in all, the same fixed, seeded sample of environments is kept in every
    per-environment array and its indices go to env_index.npy."""
    import numpy as np
    shared = shared or {}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a.nbytes // n for a in arrays.values())
    fixed = 128 * (len(arrays) + len(shared) + 1) + sum(a.nbytes for a in shared.values())   # + .npy headers
    if row_bytes * n + fixed > limit:
        keep = (limit - fixed) // (row_bytes + 8)                # + 8: the float64 index of each kept environment
        rows = np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["env_index"] = rows.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for name, a in {**arrays, **shared}.items():
        np.save(os.path.join(directory, name + ".npy"), a)


_WORKER = {}


def _reference_tree():
    """baseline/_ref (copy of the reference's Python made by baseline/build_ref.py), or None when it was not made"""
    root = os.path.join(REPO, "baseline", "_ref")
    return root if os.path.isdir(os.path.join(root, "drloco", "mujoco")) else None


def _oracle_init(n_envs, seed_base, want_reference=True):
    """per-process initialiser (like a SubprocVecEnv worker): the reference's own, unmodified
    ``Monitor(MimicWalker3dEnv())`` Python (drloco/common/utils.py:109-125) imported from baseline/_ref over
    oracle/liboracle.so when the copy exists, else the numpy restatement of the env logic (oracle/env_oracle.py)."""
    import random

    import numpy as np
    seed = seed_base + os.getpid()
    random.seed(seed)
    np.random.seed(seed % (2 ** 31))
    tree = _reference_tree() if want_reference else None
    if tree is not None:
        from baseline import ref_runner
        ref_runner.use_reference_tree(tree)
        Env, Monitor, _utils = ref_runner.load_reference()
        envs = [Monitor(Env()) for _ in range(n_envs)]
        for e in envs:
            e.reset()
        _WORKER.update(kind="reference", envs=envs, rng=np.random.default_rng(seed), n=n_envs, act=8,
                       phys=ref_runner.PHYSICS_SECONDS)
        return
    from drloco_b200.walkers import make_spec
    from oracle.env_oracle import OracleVecEnv
    from oracle.physics import OraclePhysics
    phys = [0.0]

    class TimedPhysics(OraclePhysics):
        """times the control-step integration, as ref_runner's MjSim stand-in does for the reference arm"""

        def step(self, *a):
            t0 = time.perf_counter()
            bad = super().step(*a)
            phys[0] += time.perf_counter() - t0
            return bad

    spec = make_spec()
    venv = OracleVecEnv(spec, n_envs, lambda: TimedPhysics(spec.model))
    venv.reset()
    _WORKER.update(kind="port", venv=venv, rng=np.random.default_rng(seed), n=n_envs, act=spec.act_dim, phys=phys)


def _oracle_run(n_steps):
    """n_steps control steps of this worker's envs -> (env-steps, seconds, seconds inside the physics library, kind)."""
    import numpy as np
    w = _WORKER
    p0 = w["phys"][0]
    t0 = time.perf_counter()
    if w["kind"] == "reference":
        for _ in range(n_steps):                          # DummyVecEnv.step_wait semantics (SB3 1.0), written out
            acts = w["rng"].uniform(-1, 1, (w["n"], w["act"])).astype(np.float32)
            for e, a in zip(w["envs"], acts):
                _obs, _rew, done, info = e.step(a)
                if done:
                    info["terminal_observation"] = _obs
                    e.reset()
    else:
        for _ in range(n_steps):
            w["venv"].step(w["rng"].uniform(-1, 1, (w["n"], w["act"])).astype(np.float32))
    return w["n"] * n_steps, time.perf_counter() - t0, w["phys"][0] - p0, w["kind"]


def _oracle_worker(args):
    """env-steps/s of the CPU stack in this process: (n_envs, n_steps, seed, want_reference) -> _oracle_run result"""
    n_envs, n_steps, seed, want_reference = args
    _oracle_init(n_envs, seed, want_reference)
    _oracle_run(5)
    return _oracle_run(n_steps)


PHYSICS_LIB = "oracle/liboracle.so (float64 C restatement of the MuJoCo pipeline, oracle/walker_physics.c; MuJoCo itself is not installable here)"


def cpu_baseline_single(budget_s: float = 12.0):
    """bounded single-core sample of the CPU stack (rank 0, N = 1)."""
    import multiprocessing as mp

    from oracle import physics
    physics.build()
    ctx = mp.get_context("fork")
    with ctx.Pool(1) as pool:                              # own process: the reference import chdir()s and stubs modules
        steps, secs, _p, _k = pool.apply(_oracle_worker, ((8, 30, 0, True),))
        rate = steps / secs
        n_steps = max(30, int(budget_s * rate / 8))
        steps, secs, phys, kind = pool.apply(_oracle_worker, ((8, n_steps, 1, True),))
    logic = ("the reference's unmodified MimicWalker3dEnv + Monitor Python (baseline/_ref)" if kind == "reference"
             else "numpy restatement of the reference env logic (oracle/env_oracle.py)")
    return {"value": steps / secs, "unit": "env-steps/s", "cores": 1, "kind": kind,
            "sample": f"8 envs x {n_steps} control steps, W3D RK4, random actions; {logic} over {PHYSICS_LIB}; "
                      f"{secs:.1f} s, {100 * phys / secs:.0f}% of it inside the physics library"}


def run_reference(args, emit):
    """--impl reference: the reference's path on the host cores - SubprocVecEnv = one process per env worker
    (drloco/common/utils.py:109-125), each running the reference's own Monitor(MimicWalker3dEnv()) Python from
    baseline/_ref over the physics restatement (falls back to the numpy port of the env logic when the copy is absent)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    from oracle import physics
    physics.build()
    cores = os.cpu_count() or 1
    per_proc_envs = 4
    # size each step so that steps+warmup stay within a few minutes: one "step" = 40 control steps of all envs
    ctrl_per_step = 40
    ctx = mp.get_context("fork")
    total_steps, t_total, phys_total, busy_total, kind = 0, 0.0, 0.0, 0.0, "port"
    with ctx.Pool(cores, initializer=_oracle_init, initargs=(per_proc_envs, 1000)) as pool:
        t0 = time.perf_counter()
        for k in range(args.warmup):
            pool.map(_oracle_run, [5] * cores, chunksize=1)
        per_ctrl = (time.perf_counter() - t0) / (5 * args.warmup)       # seconds per control step of all workers
        # bound the whole timed run to ~2 minutes whatever --steps is
        ctrl_per_step = max(1, min(ctrl_per_step, int(120.0 / (per_ctrl * max(1, args.steps)))))
        t0 = time.perf_counter()
        for k in range(args.steps):
            res = pool.map(_oracle_run, [ctrl_per_step] * cores, chunksize=1)
            total_steps += sum(r[0] for r in res)
            busy_total += sum(r[1] for r in res)
            phys_total += sum(r[2] for r in res)
            kind = res[0][3]
        t_total = time.perf_counter() - t0
    value = total_steps / t_total
    logic = ("the reference's unmodified MimicWalker3dEnv + Monitor Python (baseline/_ref, import stubs for gym / "
             "mujoco_py / SB3)" if kind == "reference" else
             "numpy restatement of the reference env logic (oracle/env_oracle.py; baseline/_ref absent)")
    sample = (f"{cores} processes x {per_proc_envs} envs x {ctrl_per_step} control steps per bench step; {logic}; "
              f"physics: {PHYSICS_LIB}; {100 * phys_total / max(busy_total, 1e-9):.0f}% of the workers' time inside the "
              f"physics library, the rest Python glue")
    line = {"impl": "reference", "metric": "env-steps/s incl. DeepMimic reward", "value": value, "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_total / max(1, args.steps) * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic random actions on the shipped straight-walking mocap",
            # the same workload as the CUDA arm's line (its `config`), measured on a bounded sample of it
            "config": {"workload": W3D_WORKLOAD % args.envs_per_gpu, "envs_per_gpu": args.envs_per_gpu,
                       "integrator": "rk4", "frame_skip": 5, "parallelism": f"{cores} host processes (SubprocVecEnv-like)",
                       "sample_envs": cores * per_proc_envs},
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": kind, "sample": sample,
                             "physics_fraction": phys_total / max(busy_total, 1e-9)},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--integrator", default="rk4", choices=["rk4", "euler"])
    ap.add_argument("--env-id", default=ENV_ID, choices=["StraightMimicWalker", "MimicWalker165cm65kg"],
                    help="informational runs of the other BASELINE.json configs; the headline is the default")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--stats-sync-every", type=int, default=1,
                    help="B200VecNormalize(stats_sync_every=K): exchange / merge the VecNormalize moments every K-th step "
                         "(opt-in amortisation; 1 = SB3 semantics, the headline setting)")
    ap.add_argument("--host-outputs", choices=["mapped", "copy"], default="mapped",
                    help="numpy API: kernels write the outputs into mapped pinned host memory, or one D2H copy per step")
    ap.add_argument("--pre-warmup", type=int, default=1500,
                    help="untimed steps before the W warm-up steps of the headline leg (clock / power-state ramp)")
    ap.add_argument("--no-extra", action="store_true", help="skip the time-bounded legs for BASELINE.json configs[2] / [3]")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of the headline leg, write the outputs of its last step (rank 0) as "
                         "DIR/<name>.npy (float32; the normalisation statistics float64); the inputs depend only on the "
                         "arguments, so two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the CUDA arm (--impl b200)")
    args.warmup = max(args.warmup, 3)
    # the contract is ONE JSON line on stdout: keep a private handle to the real stdout and point fd 1 at stderr so
    # that library chatter (e.g. NCCL's version banner) cannot end up in front of it
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    def emit(line):
        real_stdout.write(json.dumps(line) + "\n")
        real_stdout.flush()

    if args.impl == "reference":
        return run_reference(args, emit)

    import numpy as np
    import torch
    import torch.distributed as dist

    from drloco_b200.config import EnvConfig
    from drloco_b200.vec_env import B200MimicVecEnv, B200VecNormalize

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))
    dev = torch.device("cuda", local)
    flush = torch.empty(192 * 1024 * 1024 // 4, device=dev)                    # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def measure(env_id, n, integrator, steps, warmup, with_clocks=False, flushed_steps=0, e2e_steps=0, dump=False):
        """one workload on this rank's GPU: W warm-up steps, then K timed steps of every flavour; dump=True keeps the
        outputs of the last device-resident timed step as host arrays (out["outputs"])"""
        sampler = ClockSampler(local) if with_clocks else None
        if sampler:
            sampler.start()
        cfg = EnvConfig(env_id=env_id, integrator=integrator)
        env = B200MimicVecEnv(env_id, num_envs=n, device=f"cuda:{local}", seed=rank, cfg=cfg, env_id_offset=rank * n)
        vn = B200VecNormalize(env, distributed=world > 1, stats_sync_every=args.stats_sync_every)
        g = torch.Generator(device=dev)
        g.manual_seed(1234 + rank)
        ring = torch.rand(64, n, env.act_dim, device=dev, generator=g) * 2 - 1     # pre-generated action ring (§8d)
        out = {"exchange": vn.exchange, "frame_skip": env.spec.frame_skip, "act_dim": env.act_dim,
               "obs_dim": env.obs_dim, "lanes_per_env": env.launch_info()["lanes_per_env"]}
        vn.reset_tensor()
        if with_clocks:
            # headline leg on a box that may just have been idle: ~0.4 s of untimed steps so that clocks / power state
            # are up before the W warm-up steps (a cold box ran the first 200 steps 5 % slower; fixed count, every rank
            # takes part in each step's exchange)
            for k in range(args.pre_warmup):
                vn.step_tensor(ring[k % 64])
        for k in range(warmup):
            vn.step_tensor(ring[k % 64])
        barrier()
        env.reset_stats()
        # ---- device-resident, statistics chain overlapped (value) + per-kernel timing of the fused step kernel ----
        if sampler:
            sampler.begin()
        launches0 = env.launches + vn.launches
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        ev[0].record()
        for k in range(steps):
            a = ring[k % 64]
            vn._guard_reuse()
            vn._attach_next()
            kev[k][0].record()
            obs, rew, done = env.step_tensor(a)
            kev[k][1].record()
            # the actions of this workload do not depend on the observations: the statistics exchange + normalisation
            # kernel of step k runs on the side stream and overlaps env step k+1
            vn._normalize(obs, rew, done, wait=False)
        vn.synchronize()
        ev[1].record()
        barrier()
        ms_total = max_over_ranks(ev[0].elapsed_time(ev[1]))
        out["ms_per_step"] = ms_total / steps
        out["value"] = world * n * steps / (ms_total * 1e-3)
        out["kernel_ms"] = float(np.mean([a.elapsed_time(b) for a, b in kev]))
        out["launches"] = env.launches + vn.launches - launches0
        out["stats"] = env.stats()
        if dump:
            # what a caller of this loop holds after its last step: the env's outputs, their normalised form and the
            # running statistics they were normalised with (VecNormalize.obs_rms / ret_rms, float64).  Terminal
            # observations exist for finished environments only; the other rows are zeroed.
            fin = done.bool()
            outputs = {"obs": obs, "reward": rew, "done": done, "norm_obs": vn.norm_obs_buf,
                       "norm_reward": vn.norm_rew_buf,
                       "terminal_obs": torch.where(fin[:, None], env.terminal_obs, torch.zeros_like(env.terminal_obs))}
            out["outputs"] = {k: v.float().cpu().numpy() for k, v in outputs.items()}
            orms, rrms = vn.obs_rms, vn.ret_rms
            out["rms"] = {"obs_rms_mean": orms.mean, "obs_rms_var": orms.var,
                          "ret_rms_var": np.array([rrms.var], np.float64)}
        # ---- the same steps as a policy sees them: the normalised observation of step k before step k+1 starts ----
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        barrier()
        ev[0].record()
        for k in range(steps):
            vn.step_tensor(ring[k % 64])                 # wait=True: step -> exchange/merge/normalise, serialised
        ev[1].record()
        barrier()
        if sampler:                                      # the clocks cover the value and value_serialized regions
            sampler.end()
            out["clocks"] = sampler.stop()
        ms_ser = max_over_ranks(ev[0].elapsed_time(ev[1]))
        out["value_serialized"] = world * n * steps / (ms_ser * 1e-3)
        # ---- every step timed alone after an L2 flush (cold persistent state) ----
        if flushed_steps:
            fev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                   for _ in range(flushed_steps)]
            barrier()
            for k in range(flushed_steps):
                flush.fill_(float(k))                    # 192 MB > 126 MB L2: evicts state, mocap table and model
                fev[k][0].record()
                vn.step_tensor(ring[k % 64])
                fev[k][1].record()
            barrier()
            tf = max_over_ranks(sum(a.elapsed_time(b) for a, b in fev))
            out["value_l2_flushed"] = world * n * flushed_steps / (tf * 1e-3)
        # ---- end to end through the SB3-facing numpy API (host actions in, host obs / rew / done / infos out) ----
        if e2e_steps:
            host_actions = [np.random.default_rng(rank * 1000 + k).uniform(-1, 1, (n, env.act_dim)).astype(np.float32)
                            for k in range(8)]
            vn.host_outputs = args.host_outputs
            for k in range(10):                          # 2 eager steps, then one graph capture per buffer parity
                vn.step(host_actions[k % 8])
            barrier()
            flush.fill_(1.0)
            barrier()
            ev2 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev2[0].record()
            acc, n_term = 0.0, 0
            for k in range(e2e_steps):
                o, r, d, infos = vn.step(host_actions[k % 8])
                acc += float(r[0])
                n_term += int(d.sum())
            ev2[1].record()
            barrier()
            t2 = max_over_ranks(ev2[0].elapsed_time(ev2[1]))
            out["e2e"] = {"value": world * n * e2e_steps / (t2 * 1e-3), "unit": "env-steps/s",
                          "h2d_bytes_per_step": vn.h2d_bytes_per_step(), "d2h_bytes_per_step": vn.d2h_bytes_per_step(),
                          "steps": e2e_steps, "host_outputs": vn.host_outputs,
                          "api": "B200VecNormalize.step(host float32 actions) -> host obs, rew, done, infos (defaults)"}
        vn.close()
        return out

    n = args.envs_per_gpu
    head = measure(args.env_id, n, args.integrator, args.steps, args.warmup, with_clocks=True,
                   flushed_steps=min(args.steps, 50), e2e_steps=0 if args.no_e2e else args.steps,
                   dump=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, head["outputs"], head["rms"])
    # ---- the other GPU configurations of BASELINE.json, time-bounded (a few dozen steps each) ----
    extra = {}
    if not args.no_extra and args.env_id == ENV_ID and args.integrator == "rk4":
        n2 = 65536 // world
        m2 = measure(ENV_ID, n2, "rk4", 30, 5)
        extra["configs[2]"] = {"workload": "MimicWalker3d straight walking, 65536 envs sharded over %d GPU(s) (%d per GPU)"
                                           % (world, n2), "value": m2["value"], "value_serialized": m2["value_serialized"],
                               "ms_per_step": m2["ms_per_step"], "kernel_ms": m2["kernel_ms"], "steps": 30, "warmup": 5}
        m3 = measure(W165, 16384, "rk4", 20, 5)
        extra["configs[3]"] = {"workload": "MimicWalker165cm65kg, synthetic loco3d mocap, RSI + termination, 16384 envs "
                                           "per GPU x %d" % world, "value": m3["value"],
                               "value_serialized": m3["value_serialized"], "ms_per_step": m3["ms_per_step"],
                               "kernel_ms": m3["kernel_ms"], "steps": 20, "warmup": 5,
                               "episodes_finished": m3["stats"]["episodes"],
                               "mean_ep_len": (m3["stats"]["ep_len_sum"] / m3["stats"]["episodes"]
                                               if m3["stats"]["episodes"] else None)}

    if rank == 0:
        peaks, which = _peaks()
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        kernel_ms, stats = head["kernel_ms"], head["stats"]
        algo_bytes = ALGO_BYTES_PER_ENV_STEP if args.env_id == ENV_ID else 597.0      # SURVEY.md §8d
        algo_flop = algo_flop_per_env_step(args.env_id, args.integrator, head["frame_skip"])
        achieved_gbs = algo_bytes * n / (kernel_ms * 1e-3) / 1e9
        fp32_peak = fp32_peak_tflops(local)
        achieved_tf = algo_flop * n / (kernel_ms * 1e-3) / 1e12
        traffic, traffic_src = profiled_traffic(args.env_id, n, args.integrator)
        line = {
            "metric": "env-steps/s incl. DeepMimic reward", "value": head["value"], "unit": "env-steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic random actions U(-1,1) on the shipped straight-walking mocap, random-init (RSI) states",
            "config": {"workload": (W3D_WORKLOAD % n) if args.env_id == ENV_ID else
                                   ("MimicWalker165cm65kg on the synthetic loco3d mocap, %d envs per GPU, RSI + early "
                                    "termination (BASELINE.json configs[3])" % n),
                       "envs_per_gpu": n, "integrator": args.integrator, "frame_skip": head["frame_skip"],
                       "parallelism": f"env-sharded x{world}", "statistics_exchange": head["exchange"],
                       "stats_sync_every": args.stats_sync_every,
                       "pre_warmup": "%d untimed steps before the W warm-up steps (clock / power-state ramp)" % args.pre_warmup,
                       "l2": "value / value_serialized: the persistent env state (%.1f MB) is re-read every step as in "
                             "a real rollout; value_l2_flushed: every step re-timed alone after a 192 MB L2 flush"
                             % (n * 720 / 1e6),
                       "lanes_per_env": head["lanes_per_env"]},
            # value: statistics kernel of step k overlaps env step k+1 (legal for actions that do not depend on the
            # observations); value_serialized: what a policy sees - step, exchange + merge + normalise, next step
            "value_serialized": head["value_serialized"],
            "value_l2_flushed": head.get("value_l2_flushed"),
            "clocks": head.get("clocks"),
            "e2e": head.get("e2e"),
            "gpu_launches": head["launches"],
            "roofline": {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved_gbs / hbm_peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": which,
                         "kernel": "mimic_step_kernel", "kernel_ms": kernel_ms,
                         "note": "latency/FP32-bound by construction: %d algorithmic bytes per env-step" % algo_bytes},
            "fp32": {"achieved_tflops": achieved_tf, "peak_tflops": fp32_peak,
                     "frac": achieved_tf / fp32_peak if fp32_peak else None,
                     "peak_source": "FFMA probe kernel (8 independent chains/thread, all SMs) measured in this run; nominal 148 SM x 128 x 2 x 1.965 GHz = 74.4",
                     "algo_flop_per_env_step": algo_flop},
            "episode_stats": {"episodes": stats["episodes"], "mean_ep_len": stats["ep_len_sum"] / max(1.0, stats["episodes"]),
                              "reset_rate_per_env_step": stats["episodes"] / max(1.0, stats["env_steps"]),
                              "solver_iters_per_eval": stats["solver_iters"] / max(1.0, stats["dyn_evals"]),
                              "solver_capped_frac": stats["solver_capped"] / max(1.0, stats["dyn_evals"])},
            "extra": extra,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_single()
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
