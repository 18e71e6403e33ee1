"""Three-object tabletop auto-reset, evaluation statistics and sharding, without a GPU: the pre-drawn reset stream
against real numpy, the test oracle's auto-reset and statistics against their definitions, and the library's flag check."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import REPO
from earl_benchmark_b200 import _lib, shard_range
from earl_benchmark_b200.envs import tabletop_manipulation_3obj as tt3
from oracle import tabletop3
from tabletop3_features_oracle import Tabletop3FeaturesOracle


@pytest.mark.parametrize("seed", [0, 5, 2**32 - 1])
def test_reset_stream_rows_are_numpy_draws(seed):
    total, R = 13, 4
    full = tt3.reset_stream(seed, total, 0, total, R)
    assert full.shape == (R, total, 8) and full.dtype == np.float64
    rs = np.random.RandomState(seed)
    for e in range(R):   # bit for bit against real numpy's legacy stream
        assert np.array_equal(full[e], tt3.goal_states[0][:8] + rs.uniform(-0.3, 0.3, 8 * total).reshape(total, 8))


@pytest.mark.parametrize("parts", [[1, 12], [5, 3, 5], [4, 4, 4, 1]])
def test_reset_stream_shards_concatenate(parts):
    total, R, seed = sum(parts), 3, 9
    full = tt3.reset_stream(seed, total, 0, total, R)
    lo = 0
    for n in parts:
        assert np.array_equal(tt3.reset_stream(seed, total, lo, n, R), full[:, lo:lo + n])
        lo += n
    spans = [shard_range(1001, r, 3) for r in range(3)]
    pieces = [tt3.reset_stream(1, 1001, a, b - a, 2) for a, b in spans]
    assert np.array_equal(np.concatenate(pieces, axis=1), tt3.reset_stream(1, 1001, 0, 1001, 2))


def _actions(rs, steps, n):
    a = rs.uniform(-1.2, 1.2, (steps, n, 3)).astype(np.float32)
    a[:, : n // 2, 2] = np.where(rs.uniform(size=(steps, n // 2)) < 0.9, 1.0, -1.0)
    return a


@pytest.mark.parametrize("dense", [False, True])
@pytest.mark.parametrize("stream", [False, True])
def test_oracle_auto_reset_equals_step_then_masked_reset(dense, stream):
    n, steps, horizon = 37, 50, 7
    rs = np.random.RandomState(4)
    rows = tt3.reset_stream(3, n, 0, n, 3) if stream else None
    auto = Tabletop3FeaturesOracle(n, horizon, dense=dense, auto_reset=True, reset_rows=rows)
    man = Tabletop3FeaturesOracle(n, horizon, dense=dense, reset_rows=rows)
    assert np.array_equal(auto.reset(), man.reset())
    half = np.arange(n) % 2 == 0
    acts = _actions(rs, steps, n)
    for t in range(steps):
        if t == 3:   # stagger the episodes
            assert np.array_equal(auto.reset(mask=half), man.reset(mask=half))
        o, r, d, s = auto.step(acts[t])
        o2, r2, d2, s2 = man.step(acts[t])
        if d2.any():
            o2 = man.reset(mask=d2)
        assert np.array_equal(o, o2) and np.array_equal(r, r2) and np.array_equal(d, d2) and np.array_equal(s, s2), t
    assert d.dtype == bool and auto.num_interventions.max() > 5
    for k in ("qpos", "att", "num_interventions", "steps_since_reset", "cursor", "ep_return"):
        assert np.array_equal(getattr(auto, k), getattr(man, k)), k
    if stream:
        assert auto.cursor.max() > len(rows)   # the cursor wrapped


@pytest.mark.parametrize("dense", [False, True])
def test_oracle_eval_accumulators_equal_a_direct_sum(dense):
    n, steps = 29, 40
    rs = np.random.RandomState(8)
    orc = Tabletop3FeaturesOracle(n, 1 << 40, dense=dense)
    q0 = tabletop3.GOAL_STATES[0][:8] + rs.uniform(-0.15, 0.15, (n, 8))   # near the goal: some steps succeed
    orc.reset(init_qpos=q0)
    rews, succs = [], []
    for a in _actions(rs, steps, n):
        o, r, d, s = orc.step(a)
        rews.append(r.astype(np.float32).astype(np.float64))
        succs.append(s)
        assert np.array_equal(r, tabletop3.compute_reward(o, dense))
    ret = np.zeros(n)
    for r in rews:   # the same per-env order of additions as the device
        ret = ret + r
    succs = np.array(succs)
    assert succs.any() and not succs.all()
    want = [ret.sum(), succs[-1].sum(), succs.any(0).sum(), n]
    assert np.array_equal(orc.eval_stats(), want)
    orc.reset(mask=np.arange(n) < 10)
    assert not orc.ep_return[:10].any() and not orc.success_any[:10].any()


def test_create_accepts_the_new_flags_and_still_rejects_the_others():
    """The flag check passes and then the device check fails.  Runs where no GPU is visible: in this process on a machine
    without one, else in a child pytest that is shown none."""
    import torch
    if torch.cuda.is_available():
        test = f"{os.path.abspath(__file__)}::test_create_accepts_the_new_flags_and_still_rejects_the_others"
        r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", test], cwd=REPO,
                           env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
        return
    L = _lib.lib()
    cfg = _lib.Tt3Config()
    h = ctypes.c_void_p()
    cfg.num_envs, cfg.num_goals, cfg.episode_horizon = 4, 1, 10
    cfg.flags = _lib.FLAG_AUTO_RESET | _lib.FLAG_EVAL_STATS | _lib.FLAG_RESET_AT_GOAL | _lib.FLAG_DENSE_REWARD
    assert L.earl_tt3_create(ctypes.byref(cfg), ctypes.sizeof(cfg), ctypes.byref(h)) == -2          # EARL_ERR_CUDA
    for f in (_lib.FLAG_LIFELONG, _lib.FLAG_WIDE_INIT, _lib.FLAG_STATE_F64):
        cfg.flags = f | _lib.FLAG_AUTO_RESET
        assert L.earl_tt3_create(ctypes.byref(cfg), ctypes.sizeof(cfg), ctypes.byref(h)) == -4      # unsupported
        assert b"three-object" in L.earl_last_error()


def test_lifelong_wrapper_still_raises_and_shards_are_validated():
    from earl_benchmark_b200.wrappers.lifelong_wrapper import LifelongWrapper
    env = tt3.TabletopManipulation(num_envs=4, device="cuda:0", auto_reset=True, eval_stats=True)
    with pytest.raises(ValueError):
        LifelongWrapper(env, 10)
    with pytest.raises(ValueError):
        tt3.TabletopManipulation(num_envs=4, device="cuda:0", env_offset=3, total_envs=6)
    with pytest.raises(ValueError):
        tt3.TabletopManipulation(num_envs=4, device="cuda:0", reset_stream_rows=0)
