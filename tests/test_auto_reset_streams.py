"""Pre-drawn reset streams of the auto-reset handles (door, peg, kitchen), on the host: the native peg replay against the
env's own one-env-at-a-time draws, the shard slicing, and row e of each stream against the e-th full host reset."""
import numpy as np
import pytest

from earl_benchmark_b200 import rng
from earl_benchmark_b200.envs import kitchen, sawyer_door, sawyer_peg


def peg(seed, **kw):
    return sawyer_peg.SawyerPegV2(seed=seed, device="cuda:0", **kw)


@pytest.mark.parametrize("seed", [0, 3, 12345, 2**32 - 1])
@pytest.mark.parametrize("opts", [{}, {"wide_init": True}, {"reset_at_goal": True}])
def test_native_peg_draws_equal_draw_one(seed, opts):
    env = peg(seed, **opts)
    want = [env._draw_one() for _ in range(700)]
    rows, pos = rng.NumpyLegacyRandom(seed).peg_reset_draws(700, **opts)
    assert rows.tolist() == [r for r, _ in want]
    assert np.array_equal(pos, np.stack([p for _, p in want]))   # bit for bit, rejection loop included


def test_native_peg_draws_leave_the_stream_where_draw_one_does():
    env = peg(5, wide_init=True)
    for _ in range(300):
        env._draw_one()
    r = rng.NumpyLegacyRandom(5)
    r.peg_reset_draws(300, wide_init=True)
    assert [env._np_random.next_u32() for _ in range(8)] == [r.next_u32() for _ in range(8)]


def shards(build, total, parts):
    lo = 0
    for n in parts:
        yield lo, n, build(lo, n)
        lo += n
    assert lo == total


@pytest.mark.parametrize("reset_at_goal", [False, True])
def test_door_stream_shards_and_rows(reset_at_goal):
    total, R, seed = 37, 5, 9
    full = sawyer_door.reset_stream(seed, total, 0, total, R, reset_at_goal)
    assert full.shape == (R, total, 1) and full.dtype == np.float64
    for lo, n, part in shards(lambda lo, n: sawyer_door.reset_stream(seed, total, lo, n, R, reset_at_goal), total, [10, 20, 7]):
        assert np.array_equal(part, full[:, lo:lo + n])
    env = sawyer_door.SawyerDoorV2(seed=seed, num_envs=total, reset_at_goal=reset_at_goal, device="cuda:0")
    for e in range(R):   # row e = the e-th full reset of the host path
        assert np.array_equal(env._draw_angles(None), full[e, :, 0])


@pytest.mark.parametrize("opts", [{}, {"wide_init": True}, {"reset_at_goal": True}])
def test_peg_stream_shards_and_rows(opts):
    total, R, seed = 29, 4, 2
    rows, pos = sawyer_peg.reset_stream(seed, total, 0, total, R, **opts)
    assert rows.shape == (R, total) and pos.shape == (R, total, 3)
    for lo, n, (r, p) in shards(lambda lo, n: sawyer_peg.reset_stream(seed, total, lo, n, R, **opts), total, [13, 16]):
        assert np.array_equal(r, rows[:, lo:lo + n]) and np.array_equal(p, pos[:, lo:lo + n])
    env = peg(seed, num_envs=total, **opts)
    for e in range(R):   # the full host reset draws _draw_one for every global env in order
        want = [env._draw_one() for _ in range(total)]
        assert rows[e].tolist() == [g for g, _ in want]
        assert np.array_equal(pos[e], np.stack([p for _, p in want]))


@pytest.mark.parametrize("task", ["all_pairs", "microwave"])
def test_kitchen_stream_shards_and_rows(task):
    total, R, seed = 23, 6, 4
    config, table = kitchen.reset_stream(seed, total, 0, total, R, task)
    assert config.shape == (R, total) and config.dtype == np.uint8 and table.shape[1] == 14
    for lo, n, (c, t) in shards(lambda lo, n: kitchen.reset_stream(seed, total, lo, n, R, task), total, [5, 18]):
        assert np.array_equal(c, config[:, lo:lo + n]) and np.array_equal(t, table)
    env = kitchen.Kitchen(task=task, num_envs=total, seed=seed, device="cuda:0")
    for e in range(R):
        objs, idx = env._draw_configs(total)
        assert np.array_equal(table[config[e]], objs)
        if task == "all_pairs":
            assert np.array_equal(config[e], idx)
        else:
            assert not config[e].any() and len(table) == 1
