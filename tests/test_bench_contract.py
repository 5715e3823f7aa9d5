"""bench.py's command line: the reference arm runs on the CPU and prints one JSON line carrying
metric/value/unit/config/cpu_baseline/e2e (impl = reference); --dump-outputs writes what the timed
path returned at its last step."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT,
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stdout


def test_reference_arm_prints_contract_line():
    lines = [l for l in _run("--impl", "reference", "--steps", "100", "--warmup", "3").splitlines()
             if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_s" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0
    assert d["config"]["workload"].startswith("C1")
    cb = d["cpu_baseline"]
    # the UNMODIFIED reference classes when a reference tree is present (authoring container:
    # /root/reference; GPU box: the git-ignored install in baseline/_ref), else the oracle port
    assert cb["kind"] in ("port", "reference-classes+pf-port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["port"]["kind"] == "port" and d["port"]["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    assert _run("--impl", "reference", "--gpus", "2", "--steps", "10", "--warmup", "3", env=env).strip() == ""


def test_dump_outputs_whole_or_seeded_sample_under_64_mb(tmp_path):
    """A batch that fits is written whole; batches above 64 MB in all keep the same seeded env
    columns on every call, named in env_index.npy."""
    import types

    import numpy as np
    import torch

    import bench

    def batch(obs_dim, agents, envs, seed):
        g = torch.Generator().manual_seed(seed)
        return types.SimpleNamespace(obs_dim=obs_dim, agents=[None] * agents, num_envs=envs,
                                     obs=torch.rand(obs_dim, envs, generator=g, dtype=torch.float64),
                                     rew=torch.rand(agents, envs, generator=g, dtype=torch.float64),
                                     done=(torch.rand(envs, generator=g) < 0.5).to(torch.uint8))

    small = batch(51, 3, 4096, 1)
    bench._dump_outputs(str(tmp_path / "small"), {"": small})
    assert sorted(os.listdir(tmp_path / "small")) == ["done.npy", "obs.npy", "reward.npy"]
    np.testing.assert_array_equal(np.load(tmp_path / "small" / "obs.npy"), small.obs.numpy())
    np.testing.assert_array_equal(np.load(tmp_path / "small" / "reward.npy"), small.rew.numpy())
    done = np.load(tmp_path / "small" / "done.npy")
    assert done.dtype == np.float32 and np.array_equal(done, small.done.numpy())

    big = {"c1_": batch(51, 3, 262144, 2), "c3_": batch(470, 100, 16384, 3)}
    for d in ("a", "b"):
        bench._dump_outputs(str(tmp_path / d), big)
    files = sorted(os.listdir(tmp_path / "a"))
    assert len(files) == 8
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10 ** 6
    for f in files:
        np.testing.assert_array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
    for prefix, env in big.items():
        idx = np.load(tmp_path / "a" / f"{prefix}env_index.npy").astype(np.int64)
        assert 0 < len(idx) < env.num_envs and np.all(np.diff(idx) > 0)
        np.testing.assert_array_equal(np.load(tmp_path / "a" / f"{prefix}obs.npy"), env.obs.numpy()[:, idx])
        np.testing.assert_array_equal(np.load(tmp_path / "a" / f"{prefix}reward.npy"), env.rew.numpy()[:, idx])


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_path_repeat_run_to_run(tmp_path):
    """Two runs with the same arguments step the same seeded inputs and dump the same
    observations, rewards and done flags of the last timed step."""
    import numpy as np
    args = ("--gpus", "1", "--steps", "5", "--warmup", "3", "--no-cpu-baseline", "--no-extra")
    for d in ("a", "b"):
        lines = [l for l in _run(*args, "--dump-outputs", str(tmp_path / d)).splitlines() if l.startswith("{")]
        assert json.loads(lines[-1])["steps"] == 5
    shapes = {"obs.npy": (51, 4096), "reward.npy": (3, 4096), "done.npy": (4096,)}
    assert sorted(os.listdir(tmp_path / "a")) == sorted(shapes)
    for f, shape in shapes.items():
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.shape == shape and a.dtype in (np.float32, np.float64) and np.isfinite(a).all()
        np.testing.assert_array_equal(a, b)
