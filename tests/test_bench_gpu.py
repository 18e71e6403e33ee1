"""bench.py on the device: `--steps K` times exactly K steps, and `--dump-outputs` writes what the last timed step computed
(checked against a replay of the same seeded inputs through the public API)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import REPO

pytestmark = pytest.mark.gpu


def test_dump_outputs_is_the_last_timed_step_of_a_replay(tmp_path):
    import bench
    import earl_benchmark_b200 as eb
    n, steps, warmup = 1 << 16, 5, 3
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--num-envs", str(n), "--steps", str(steps),
                          "--warmup", str(warmup), "--no-door", "--no-hbm-check", "--no-cpu-baseline",
                          "--dump-outputs", str(out)], cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-4000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["gpu_launches"] == steps and line["e2e"]["steps"] == steps
    got = {k: np.load(out / f"{k}.npy") for k in ("obs", "reward", "done")}
    assert sorted(os.listdir(out)) == ["done.npy", "obs.npy", "reward.npy"]
    assert all(a.dtype == np.float32 for a in got.values())
    assert got["obs"].shape == (n, 12) and got["reward"].shape == (n,) and got["done"].shape == (n,)

    # the bench's inputs: reset, W warm-up steps, one K-step priming block, the K timed steps (every block starts at action 0)
    train, _ = eb.EARLEnvs("tabletop_manipulation", reward_type="sparse", num_envs=n, device="cuda:0", seed=0,
                           train_horizon=bench.TRAIN_HORIZON, goal_stream_rows=2).get_envs()
    train.reset()
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(1234)
    actions = torch.rand((bench.ACTION_RING, n, 3), generator=gen, device="cuda:0", dtype=torch.float32) * 2 - 1
    obs = torch.empty((bench.OUT_RING, n, 12), device="cuda:0")
    rew = torch.empty((bench.OUT_RING, n), device="cuda:0")
    done = torch.empty((bench.OUT_RING, n), device="cuda:0", dtype=torch.uint8)
    for k in (warmup, steps, steps):
        train.env.rollout_into(actions, k, obs, rew, done)
    last = steps - 1
    assert np.array_equal(got["obs"], obs[last].cpu().numpy())
    assert np.array_equal(got["reward"], rew[last].cpu().numpy())
    assert np.array_equal(got["done"], done[last].float().cpu().numpy())
