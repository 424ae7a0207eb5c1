"""bench.py contract on the CPU: the reference arm (`--impl reference`) prints exactly one JSON line with the keys the
driver reads, on the CUDA arm's metric / unit / workload; without a GPU the CUDA arm must fail loudly (no CPU path)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*argv, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True,
                          timeout=300, cwd=ROOT, env={**os.environ, **(env or {})})


def test_reference_arm_line():
    p = _run("--impl", "reference", "--steps", "2", "--warmup", "1")
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [x for x in p.stdout.splitlines() if x.strip()]
    assert len(lines) == 1                                            # ONE JSON line on stdout, nothing else
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env-steps/s incl. DeepMimic reward"
    assert d["unit"] == "env-steps/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["value"] > 100 and d["steps"] == 2 and d["gpu_launches"] == 0
    assert "BASELINE.json configs[1]" in d["config"]["workload"] and d["config"]["envs_per_gpu"] == 4096
    cb = d["cpu_baseline"]
    # "reference": the reference's own Python (baseline/_ref, made by baseline/build_ref.py) ran; "port": the numpy
    # restatement stood in because the copy is absent.  Either way the sample names the library that did the physics.
    have_ref = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "drloco", "mujoco"))
    assert cb["kind"] == ("reference" if have_ref else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and "liboracle.so" in cb["sample"]
    assert 0.0 < cb["physics_fraction"] < 1.0
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    p = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--gpus", "2", env={"RANK": "1", "WORLD_SIZE": "2"})
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_steps_must_be_positive():
    p = _run("--impl", "reference", "--steps", "0", "--warmup", "1")
    assert p.returncode != 0 and p.stdout.strip() == ""


def test_write_outputs_samples_the_same_environments(tmp_path):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    n = 1000
    arrays = {"obs": np.arange(n * 29, dtype=np.float32).reshape(n, 29), "reward": np.arange(n, dtype=np.float32)}
    bench.write_outputs(str(tmp_path / "all"), arrays)
    assert sorted(os.listdir(tmp_path / "all")) == ["obs.npy", "reward.npy"]
    np.testing.assert_array_equal(np.load(tmp_path / "all" / "obs.npy"), arrays["obs"])
    limit = 40_000                                                    # below the 120 kB of the arrays
    mean = np.linspace(-1, 1, 29)                                     # shared: written whole, counted in the limit
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), arrays, {"obs_rms_mean": mean}, limit=limit)
        files = sorted(os.listdir(tmp_path / d))
        assert files == ["env_index.npy", "obs.npy", "obs_rms_mean.npy", "reward.npy"]
        assert sum(os.path.getsize(tmp_path / d / f) for f in files) <= limit
    for f in ("env_index.npy", "obs.npy", "reward.npy"):              # a fixed sample: the same rows every time
        np.testing.assert_array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
    idx = np.load(tmp_path / "a" / "env_index.npy").astype(np.int64)
    assert len(idx) > 100 and np.all(np.diff(idx) > 0)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "obs.npy"), arrays["obs"][idx])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "reward.npy"), arrays["reward"][idx])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "obs_rms_mean.npy"), mean)


@pytest.mark.gpu
def test_dump_outputs_repeat_bit_for_bit(tmp_path):
    """two runs with the same arguments dump identical outputs, and the outputs belong to one step: the normalised
    ones follow from the raw ones through the final running statistics (SB3 VecNormalize: merge, then normalise)"""
    import numpy as np
    lines = []
    for d in ("a", "b"):
        p = _run("--steps", "4", "--warmup", "3", "--pre-warmup", "0", "--envs-per-gpu", "512", "--no-cpu-baseline",
                 "--no-e2e", "--no-extra", "--dump-outputs", str(tmp_path / d))
        assert p.returncode == 0, p.stderr[-2000:]
        lines.append(json.loads(p.stdout))
    assert lines[0]["steps"] == 4 and lines[0]["gpu_launches"] == 2 * 4    # step kernel + statistics kernel per step
    names = ["done", "norm_obs", "norm_reward", "obs", "reward", "terminal_obs"]
    stats = ["obs_rms_mean", "obs_rms_var", "ret_rms_var"]
    assert sorted(f[:-4] for f in os.listdir(tmp_path / "a")) == sorted(names + stats)
    g = {}
    for name in names + stats:
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == (np.float32 if name in names else np.float64) and np.all(np.isfinite(a)), name
        assert len(a) == (512 if name in names else 29 if name.startswith("obs") else 1), name
        np.testing.assert_array_equal(a, b, err_msg=name)
        g[name] = a
    assert g["obs"].shape == g["norm_obs"].shape == g["terminal_obs"].shape == (512, 29)
    # the kernel's arithmetic (csrc/vecnorm.cu): float32 mean and 1/sqrt(var + eps), clip at 10; eps = 1e-8 as a float
    eps = np.float64(np.float32(1e-8))
    inv = (1.0 / np.sqrt(g["obs_rms_var"] + eps)).astype(np.float32)
    want = np.clip((g["obs"] - g["obs_rms_mean"].astype(np.float32)) * inv, -10, 10)
    np.testing.assert_allclose(g["norm_obs"], want, rtol=0, atol=1e-5)
    want = np.clip(g["reward"] * np.float32(1.0 / np.sqrt(g["ret_rms_var"][0] + eps)), -10, 10)
    np.testing.assert_allclose(g["norm_reward"], want, rtol=0, atol=1e-5)
    done = g["done"].astype(bool)
    assert set(np.unique(g["done"])) <= {0.0, 1.0}
    assert not g["terminal_obs"][~done].any() and np.all(np.abs(g["terminal_obs"][done]).sum(axis=1) > 0)


def test_cuda_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    p = _run("--steps", "1", "--warmup", "1", "--no-cpu-baseline")
    assert p.returncode != 0 and p.stdout.strip() == ""               # no number is printed from a CPU fallback
