"""Parity of the CUDA tabletop path (through the C ABI) against the pinned CPU oracle, the golden
outputs of the unmodified reference, and the shipped demonstrations.  Needs a GPU: `-m gpu`.

Bars (BASELINE.json north_star): observations bit-exact against the oracle (fp64 arithmetic, one rounding
to fp32); integer bookkeeping bit-exact; sparse reward bit-exact outside 1e-5 of the 0.2 threshold (here it
is bit-exact everywhere, the band is only used against numpy-2-evaluated reference rewards); dense reward
within 2e-6 relative (fp32 output of an fp64 evaluation).
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import earl_benchmark_b200 as eb  # noqa: E402
from earl_benchmark_b200 import demos  # noqa: E402
from earl_benchmark_b200.envs.tabletop_manipulation import TabletopManipulation  # noqa: E402
from earl_benchmark_b200.wrappers.persistent_state_wrapper import PersistentStateWrapper  # noqa: E402
from oracle import loader  # noqa: E402
from oracle.loader import GOAL_STATES, TabletopOracle  # noqa: E402

DEV = "cuda:0"
BAND = 1e-5


def make(n, horizon=10**9, **kw):
    kw.setdefault("reward_type", "sparse")
    return PersistentStateWrapper(TabletopManipulation(num_envs=n, device=DEV, **kw), horizon)


def goal_row(obs):
    d = np.abs(GOAL_STATES[None, :, 2:4] - obs[:, None, 8:10]).sum(-1)
    return d.argmin(1)


def actions(n, steps, seed, grip_bias=0.0):
    rs = np.random.RandomState(seed)
    a = rs.uniform(-1.2, 1.2, (steps, n, 3)).astype(np.float32)
    a[..., 2] += grip_bias
    return a


def np_(t):
    return t.detach().cpu().numpy()


# ---------------------------------------------------------------------------------------- demos + goldens

@pytest.mark.parametrize("state_dtype", ["float32", "float64"])
@pytest.mark.parametrize("direction", ["forward", "reverse"])
def test_demo_transitions(golden_dir, direction, state_dtype):
    """All shipped tabletop transitions in ONE launch: == reference step() bit for bit."""
    d = demos.load("tabletop_manipulation", direction)
    ref = np.load(os.path.join(golden_dir, "tabletop_ref_demo_replay.npz"))
    n = len(d["actions"])
    env = make(n, state_dtype=state_dtype)
    env.reset()
    o = d["observations"]
    rows = env._goal_rows_for(o[:, 6:].astype(np.float64))
    env.set_state(qpos=o[:, :4].astype(np.float64), attached=(o[:, 4] == 0), goal_row=rows)
    assert np.array_equal(np_(env.get_obs()), o)
    obs, rew, done, info = env.step(torch.from_numpy(d["actions"]).to(DEV))
    obs, rew = np_(obs), np_(rew)
    assert np.array_equal(obs, ref[f"{direction}_ref_next_obs"])
    assert np.array_equal(rew.astype(np.float64), ref[f"{direction}_ref_reward"])
    assert np.abs(obs - d["next_observations"]).max() <= 2.4e-7     # stored fp32 snapshot of fp64 state: 1 ulp
    assert np.array_equal(obs[:, 4:], d["next_observations"][:, 4:])  # attach flags and goals exact
    assert np.array_equal(rew, d["rewards"][:, 0])                    # 100 % sparse-reward agreement
    assert np.array_equal(np_(info["success"]), d["rewards"][:, 0] > 0)
    assert not done.any() and env.total_steps == 1


def _replay_golden(g, prefix, horizon, dense=False, wide=False, custom_init=False, reset_at_goal=False):
    g = {k[len(prefix) + 1:]: g[k] for k in g.files if k.startswith(prefix + "_")}
    n = len(g["actions"])
    env = make(1, horizon, reward_type="dense" if dense else "sparse", wide_init_distr=wide,
               reset_at_goal=reset_at_goal, state_dtype="float64")
    acts = torch.from_numpy(g["actions"]).to(DEV)

    def do_reset(obs_row, q):
        return np_(env.reset(goal_rows=goal_row(obs_row), init_qpos=q if custom_init else None))

    o = do_reset(g["obs"][0:1], g["qpos"][0:1])
    assert np.array_equal(o[0], g["obs"][0])
    resets = 1
    for t in range(n):
        ob, rw, dn, info = env.step(acts[t:t + 1])
        ob, rw, dn, sc = np_(ob), np_(rw), np_(dn), np_(info["success"])
        if not g["reset_after"][t]:
            assert np.array_equal(ob[0], g["obs"][t + 1]), (prefix, t)
        nrm = np.linalg.norm((ob[0, 2:4] - ob[0, 8:10]) if wide else (ob[0, :4] - ob[0, 6:10]))
        if abs(nrm - 0.2) > BAND:
            assert bool(sc[0]) == bool(g["success"][t]), (prefix, t)
            if not dense:
                assert rw[0] == g["reward"][t], (prefix, t)
        if dense:
            assert abs(rw[0] - g["reward"][t]) <= 2e-6 * max(1.0, abs(g["reward"][t])), (prefix, t)
        assert bool(dn[0]) == bool(g["done"][t]), (prefix, t)
        if g["reset_after"][t]:
            o = do_reset(g["obs"][t + 1:t + 2], g["qpos"][t + 1:t + 2])
            assert np.array_equal(o[0], g["obs"][t + 1]), (prefix, t)
            resets += 1
    assert env.total_steps == g["total_steps"][-1]
    assert int(env.num_interventions[0]) == resets
    return g


@pytest.fixture(scope="module")
def rollouts(golden_dir):
    return np.load(os.path.join(golden_dir, "tabletop_ref_rollouts.npz"))


def test_golden_sparse_train_rollout(rollouts):
    """4,096-step reference trajectory (horizon 1000, 4 resets): every observation bit-exact (fp64 state)."""
    _replay_golden(rollouts, "sparse_train", 1000)


def test_golden_dense_rollout(rollouts):
    _replay_golden(rollouts, "dense_train", 700, dense=True)


def test_golden_wide_init_rollout(rollouts):
    _replay_golden(rollouts, "wide_train", 250, wide=True, custom_init=True)


def test_golden_reset_at_goal_rollout(rollouts):
    # reset_at_goal: the reset kernel itself places the env at its drawn goal (no init_qpos passed)
    _replay_golden(rollouts, "resetgoal_train", 300, reset_at_goal=True)


def test_golden_no_reset_after_done(rollouts):
    g = _replay_golden(rollouts, "noreset_train", 100)
    assert g["done"][99:].all()


def test_golden_lifelong(golden_dir):
    """LifelongWrapper on device vs the reference: seed-7 `random` stream drives resets AND goal swaps."""
    g = np.load(os.path.join(golden_dir, "tabletop_ref_lifelong.npz"))
    freq, horizon, seed = int(g["goal_change_frequency"]), int(g["train_horizon"]), int(g["seed"])
    env = eb.EARLEnvs("tabletop_manipulation", reward_type="sparse", setup_as_lifelong_learning=True,
                      train_horizon=horizon, goal_change_frequency=freq, seed=seed, state_dtype="float64",
                      device=DEV, goal_stream_rows=128).get_envs()
    acts = torch.from_numpy(g["actions"]).to(DEV)
    o = np_(env.reset())
    assert np.array_equal(o[0], g["obs"][0])
    for t in range(len(acts)):
        ob, rw, dn, _ = env.step(acts[t:t + 1])
        assert float(rw[0]) == g["reward"][t] and bool(dn[0]) == bool(g["done"][t]), t
        if g["reset_after"][t]:
            ob = env.reset()
        assert np.array_equal(np_(ob)[0], g["obs"][t + 1]), t
        assert float(env.lifelong_return[0]) == g["lifelong_return"][t]
    assert int(env.num_interventions[0]) == int(g["num_interventions"][-1]) + int(g["reset_after"][-1])


def test_shared_goal_stream_order(golden_dir):
    """16 envs, 3 resets: goals equal those of 16 reference envs sharing the global `random` stream."""
    g = np.load(os.path.join(golden_dir, "tabletop_ref_streams.npz"))["shared_stream_seed11_16envs_3resets"]
    env = make(16, seed=11)
    for r in range(3):
        o = np_(env.reset())
        assert np.array_equal(goal_row(o), g[r])
    assert np_(env.num_interventions).tolist() == [3] * 16


# ---------------------------------------------------------------------------------------- random batched parity

@pytest.mark.parametrize("n", [1, 31, 33, 257, 100003])
@pytest.mark.parametrize("state_dtype", ["float32", "float64"])
def test_random_rollout_vs_oracle(n, state_dtype):
    """Ragged batch sizes, random actions (some out of range), horizon firing mid-run: bit-exact vs oracle."""
    steps, horizon = 60, 41
    env = make(n, horizon, state_dtype=state_dtype, seed=n)
    orc = TabletopOracle(n, horizon, state_f32=(state_dtype == "float32"))
    o = np_(env.reset())
    rows = goal_row(o)
    assert np.array_equal(orc.reset(rows), o)
    acts = actions(n, steps, seed=n, grip_bias=0.3)
    # start half of the envs next to the mug so attach / drag / clip paths are busy
    q = np.tile([0.0, 0.0, 2.5, 0.0], (n, 1))
    q[::2, 0] = 2.3
    q = q.astype(np.float32).astype(np.float64)  # representable in either state dtype
    env.set_state(qpos=q)
    orc.qpos[:] = q
    for t in range(steps):
        ob, rw, dn, info = env.step(torch.from_numpy(acts[t]).to(DEV))
        o2, r2, d2, s2 = orc.step(acts[t])
        assert np.array_equal(np_(ob), o2), t
        assert np.array_equal(np_(rw).astype(np.float64), r2), t
        assert np.array_equal(np_(dn), d2.astype(bool)), t
        assert np.array_equal(np_(info["success"]), s2.astype(bool)), t
    if n >= 100003:  # the run exercised attach and the workspace clip
        assert (orc.attached != 0).any() and (np.abs(orc.qpos) >= 2.79999).any()
    total, interv, since, _ = env.env._counters()
    assert total == steps == orc.total_steps[0]
    assert np.array_equal(np_(since).astype(np.int64), orc.steps_since_reset)
    assert np.array_equal(np_(interv), orc.num_interventions)
    snap = env.get_state()
    if state_dtype == "float64":
        assert np.array_equal(snap["qpos"], orc.qpos)
    assert np.array_equal(snap["attached"], orc.attached != 0)


def test_full_size_batch_vs_oracle():
    """BASELINE config 2 size (1,048,576 envs): direct comparison with the oracle + order-independence."""
    n, steps = 1 << 20, 6
    env = make(n, 4)
    orc = TabletopOracle(n, 4, state_f32=True)
    orc.reset(goal_row(np_(env.reset())))
    acts = actions(n, steps, seed=99, grip_bias=0.5)
    rs = np.random.RandomState(5)
    q = rs.uniform(-2.8, 2.8, (n, 4)).astype(np.float32).astype(np.float64)
    q[::3, 2:4] = q[::3, 0:2] + 0.1  # a third of the envs start within the attach radius
    q = np.clip(q, -2.8, 2.8).astype(np.float32).astype(np.float64)
    env.set_state(qpos=q)
    orc.qpos[:] = q
    perm = rs.permutation(n)
    env_p = make(n, 4)
    env_p.reset(goal_rows=goal_row(orc.get_obs())[perm])
    env_p.set_state(qpos=q[perm])
    for t in range(steps):
        ob, rw, dn, _ = env.step(torch.from_numpy(acts[t]).to(DEV))
        o2, r2, d2, _ = orc.step(acts[t])
        assert np.array_equal(np_(ob), o2) and np.array_equal(np_(rw).astype(np.float64), r2)
        assert np.array_equal(np_(dn), d2.astype(bool))
        obp, rwp, _, _ = env_p.step(torch.from_numpy(acts[t][perm]).to(DEV))
        assert torch.equal(obp, ob[torch.from_numpy(perm).to(DEV)])  # envs are independent of their index
    assert (orc.attached != 0).mean() > 0.05 and np_(dn).all()


def test_f32_state_drift_is_bounded():
    """fp32 device state vs the reference's fp64 state over a long open-loop rollout: one-step error is one
    fp32 rounding (<=1.2e-7 * |x|), so drift stays far inside north_star's 1e-4."""
    n, steps = 512, 3000
    env = make(n, seed=1)
    orc = TabletopOracle(n, 10**9, state_f32=False)
    orc.reset(goal_row(np_(env.reset())))
    acts = actions(n, steps, seed=3)
    acts[..., 2] = -1.0  # no attach decisions, pure integration
    dev = torch.from_numpy(acts).to(DEV)
    for t in range(steps):
        ob, _, _, _ = env.step(dev[t])
        orc.step(acts[t])
    err = np.abs(np_(ob)[:, :4].astype(np.float64) - orc.qpos).max()
    assert err < 1e-4, err


# ---------------------------------------------------------------------------------------- features

def test_dense_reward_and_compute_reward_vs_oracle():
    n = 5000
    env = make(n, reward_type="dense")
    env.reset()
    rs = np.random.RandomState(0)
    q = rs.uniform(-2.8, 2.8, (n, 4))
    q[::4, 2:4] = np.array([0.0, 2.0]) + rs.normal(0, 0.05, (len(q[::4]), 2))
    env.set_state(qpos=q, goal_row=2)
    a = actions(n, 1, 7)[0]
    ob, rw, _, info = env.step(torch.from_numpy(a).to(DEV))
    ob = np_(ob)
    want = np.zeros(n)
    ws = np.zeros(n, np.uint8)
    loader.lib().earl_oracle_tt_reward(n, np.ascontiguousarray(ob), 1, 0, want, ws)
    assert np.abs(np_(rw) - want).max() <= 2e-6 * np.abs(want).max()
    assert np.array_equal(np_(info["success"]), ws.astype(bool))
    # compute_reward / is_successful on caller-supplied observations (device and host inputs)
    r2 = env.compute_reward(torch.from_numpy(ob).to(DEV))
    assert np.abs(np_(r2) - want).max() <= 2e-6 * np.abs(want).max()
    assert np.array_equal(env.is_successful(ob), ws.astype(bool))
    sparse = make(n)
    sparse.reset()
    loader.lib().earl_oracle_tt_reward(n, np.ascontiguousarray(ob), 0, 0, want, ws)
    assert np.array_equal(sparse.compute_reward(ob).astype(np.float64), want)
    wide = make(n, wide_init_distr=True)
    wide.reset(init_qpos=q)
    loader.lib().earl_oracle_tt_reward(n, np.ascontiguousarray(ob), 0, 1, want, ws)
    assert np.array_equal(wide.is_successful(ob), ws.astype(bool)) and ws.sum() > 0


def test_auto_reset_matches_manual_reset():
    """In-kernel reset at the horizon == the user calling reset() after done (goal stream order included)."""
    n, horizon, steps = 1000, 17, 70
    auto = make(n, horizon, auto_reset=True, seed=4)
    manual = make(n, horizon, seed=4)
    oa, om = auto.reset(), manual.reset()
    assert torch.equal(oa, om)
    acts = torch.from_numpy(actions(n, steps, 11, 0.4)).to(DEV)
    for t in range(steps):
        oa, ra, da, _ = auto.step(acts[t])
        om, rm, dm, _ = manual.step(acts[t])
        assert torch.equal(ra, rm) and torch.equal(da, dm)
        if bool(dm.all()):
            om = manual.reset()
        assert torch.equal(oa, om), t
    assert torch.equal(auto.num_interventions, manual.num_interventions)
    assert int(auto.num_interventions[0]) == 1 + steps // horizon
    ra_goal = make(n, horizon, auto_reset=True, reset_at_goal=True, seed=4)
    o = ra_goal.reset()
    assert torch.equal(o[:, :4], o[:, 6:10])  # reset_at_goal: env starts at its goal
    for t in range(horizon):
        o, _, d, _ = ra_goal.step(acts[t])
    assert bool(d.all()) and torch.equal(o[:, :4], o[:, 6:10])


def test_masked_reset_and_counters():
    n = 300
    env = make(n, 50)
    env.reset()
    acts = torch.from_numpy(actions(n, 10, 2)).to(DEV)
    for t in range(10):
        env.step(acts[t])
    mask = torch.zeros(n, dtype=torch.bool, device=DEV)
    mask[::3] = True
    before = np_(env.get_obs())
    o = np_(env.reset(mask=mask))
    m = np_(mask)
    assert np.array_equal(o[~m, :6], before[~m, :6])            # untouched envs keep their state
    assert np.array_equal(o[m, :4], np.tile([0, 0, 2.5, 0], (m.sum(), 1)))
    assert np.array_equal(np_(env.num_interventions), 1 + m.astype(np.int64))
    assert np.array_equal(np_(env.steps_since_reset), np.where(m, 0, 10))
    assert env.total_steps == 10


def test_reset_goal_custom_and_stream():
    n = 64
    env = make(n, seed=9)
    o0 = np_(env.reset())
    custom = np.array([0.0, 0.0, 1.25, -0.5, -1.0, -1.0])
    env.reset_goal(custom)
    o = np_(env.get_obs())
    assert np.array_equal(o[:, 6:], np.tile(custom.astype(np.float32), (n, 1))) and np.array_equal(o[:, :6], o0[:, :6])
    assert np.array_equal(env.goal, np.tile(custom, (n, 1)))
    env.reset_goal()  # next draw of every env's stream
    from earl_benchmark_b200 import rng
    stream = rng.PyRandom(9).tabletop_goal_rows(2 * n).reshape(2, n)
    assert np.array_equal(goal_row(np_(env.get_obs())), stream[1])
    nxt = env.get_next_goal()  # third draw, returned but not installed
    stream3 = rng.PyRandom(9).tabletop_goal_rows(3 * n).reshape(3, n)
    assert np.array_equal(nxt[:, 2:4], GOAL_STATES[stream3[2], 2:4])
    assert np.array_equal(goal_row(np_(env.get_obs())), stream[1])


def test_snapshot_roundtrip():
    n = 1234
    env = make(n, 30, seed=2)
    env.reset()
    acts = torch.from_numpy(actions(n, 40, 5, 0.4)).to(DEV)
    for t in range(20):
        env.step(acts[t])
    snap = env.get_state()
    ref = [tuple(x.clone() for x in env.step(acts[t])[:3]) for t in range(20, 40)]
    env2 = make(n, 30, seed=2)
    env2.set_state(snap)
    assert env2.total_steps == 20
    for t in range(20, 40):
        o, r, d, _ = env2.step(acts[t])
        assert torch.equal(o, ref[t - 20][0]) and torch.equal(r, ref[t - 20][1]) and torch.equal(d, ref[t - 20][2])


def test_host_buffer_path_equals_device_path():
    n = 4099
    dev_env, host_env = make(n, 9), make(n, 9)
    dev_env.reset(), host_env.reset()
    acts = actions(n, 12, 8, 0.3)
    for t in range(12):
        o, r, d, i = dev_env.step(torch.from_numpy(acts[t]).to(DEV))
        ho, hr, hd, hi = host_env.step(acts[t])  # numpy in -> numpy out, copies inside the call
        assert isinstance(ho, np.ndarray)
        assert np.array_equal(ho, np_(o)) and np.array_equal(hr, np_(r)) and np.array_equal(hd, np_(d))
        assert np.array_equal(hi["success"], np_(i["success"]))
    pinned = torch.from_numpy(acts[0]).pin_memory()
    ho, _, _, _ = host_env.step(pinned)
    assert ho.shape == (n, 12) and host_env.total_steps == 13


def test_rollout_equals_repeated_step():
    n, k, steps = 777, 5, 13
    a, b = make(n, 7), make(n, 7)
    a.reset(), b.reset()
    acts = torch.from_numpy(actions(n, k, 21, 0.3)).to(DEV)
    obs = torch.empty((4, n, 12), device=DEV)
    rew = torch.empty((4, n), device=DEV)
    done = torch.empty((4, n), dtype=torch.uint8, device=DEV)
    a.rollout_into(acts, steps, obs, rew, done)
    for t in range(steps):
        o, r, d, _ = b.step(acts[t % k])
        if t >= steps - 4:
            assert torch.equal(obs[t % 4], o) and torch.equal(rew[t % 4], r) and torch.equal(done[t % 4].bool(), d)
    assert a.total_steps == b.total_steps == steps


def test_eval_stats():
    n, horizon = 2000, 25
    loader_ = eb.EARLEnvs("tabletop_manipulation", reward_type="sparse", num_envs=n, eval_horizon=horizon, device=DEV)
    _, ev = loader_.get_envs()
    ev.reset()
    rs = np.random.RandomState(1)
    q = np.tile([0.0, 0.0, 2.5, 0.0], (n, 1))
    goals = np_(ev.get_obs())[:, 6:10].astype(np.float64)
    q[::2] = goals[::2] + rs.normal(0, 0.08, (n // 2, 4))  # half of the envs start near success
    ev.set_state(qpos=np.clip(q, -2.8, 2.8))
    acts = torch.from_numpy((0.3 * actions(n, horizon, 3)).astype(np.float32)).to(DEV)
    ret = np.zeros(n)
    anyv = np.zeros(n, bool)
    for t in range(horizon):
        o, r, d, i = ev.step(acts[t])
        ret += np_(r)
        anyv |= np_(i["success"])
    last = np_(i["success"])
    s = np_(ev.eval_stats())
    assert s[3] == n and s[0] == ret.sum() and s[1] == last.sum() and s[2] == anyv.sum() and ret.sum() > 0
    from earl_benchmark_b200.distributed import all_reduce_eval_stats
    res = all_reduce_eval_stats(ev.eval_stats())
    assert abs(res["mean_return"] - ret.mean()) < 1e-12 and res["num_envs"] == n
    ev.reset()
    assert np_(ev.eval_stats())[:3].tolist() == [0.0, 0.0, 0.0]


def test_invalid_arguments_fail_loudly():
    from earl_benchmark_b200 import _lib
    env = make(8)
    env.reset()
    with pytest.raises(ValueError):
        env.step(torch.zeros((7, 3), device=DEV))
    with pytest.raises(_lib.EarlError):
        TabletopManipulation(num_envs=0, device=DEV, reward_type="sparse").reset()
    with pytest.raises(_lib.EarlError):  # misaligned observation buffer
        buf = torch.empty(8 * 12 + 1, device=DEV)[1:].view(8, 12)
        env.step(torch.zeros((8, 3), device=DEV), out=(buf, env._reward, env._done, env._success))


def test_config1_full_reset_free_horizon():
    """BASELINE.json configs[0] at its true size (SURVEY 8(d) config 1): sparse reward, default train horizon 200,000,
    200,000 random-action steps in ONE device rollout.  `done` is first True at step index 199,999, total_steps ==
    200000, num_interventions == 1, and every observation / reward of the run is bit-exact against the checker."""
    n, steps = 8, 200000
    train, _ = eb.EARLEnvs("tabletop_manipulation", reward_type="sparse", num_envs=n, device=DEV, seed=0,
                           state_dtype="float64").get_envs()
    assert train._episode_horizon == steps
    o0 = np_(train.reset())
    orc = TabletopOracle(n, steps, state_f32=False)
    assert np.array_equal(orc.reset(goal_row(o0)), o0)
    acts = np.random.RandomState(0).uniform(-1, 1, (steps, n, 3)).astype(np.float32)
    acts[:, : n // 2, 2] = np.abs(acts[:, : n // 2, 2])          # half of the envs keep the gripper closed: they drag the mug
    obs = torch.empty((steps, n, 12), device=DEV)
    rew = torch.empty((steps, n), device=DEV)
    done = torch.empty((steps, n), dtype=torch.uint8, device=DEV)
    train.rollout_into(torch.from_numpy(acts).to(DEV), steps, obs, rew, done)
    obs, rew, done = np_(obs), np_(rew), np_(done)
    assert not done[:-1].any() and done[-1].all()                 # first True at index 199,999
    assert train.total_steps == steps and (np_(train.num_interventions) == 1).all()
    dragged = 0
    for t in range(steps):
        o2, r2, d2, _ = orc.step(acts[t])
        if not (np.array_equal(obs[t], o2) and np.array_equal(rew[t].astype(np.float64), r2)):
            raise AssertionError(f"mismatch at step {t}")
        dragged += int((orc.attached != 0).sum())
    assert bool(d2.all()) and dragged > steps                     # the attach / drag path was busy
    assert np.array_equal(train.get_state()["qpos"], orc.qpos)    # fp64 state after 200,000 steps, bit for bit


def test_f32_state_against_the_fp64_reference_over_the_benchmarked_horizon():
    """VERDICT r1 weak #8: every bench number runs with the state STORED as fp32 (the 113-B layout) while the reference keeps
    fp64 qpos.  One step from an fp32-representable state is bit-exact, but over the benchmarked 200,000-step reset-free
    horizon an attach decision (||fist - mug|| < 0.4) or a success test can flip on a 1-ulp state difference and the two
    trajectories then part for good.  Measured here on 2,048 envs x 200,000 random-action steps (gripper closing half of the
    time, so the mug is grabbed, dragged and dropped all along): the fraction of envs whose attached-flag or sparse-reward
    SEQUENCE ever differs from the fp64 checker's, the first step at which that happens, and the state error of the envs
    that never diverged.  Decision flips are rare but real -- which is why `state_dtype='float64'` exists and is the mode the
    bit-exact claims are made for (test_config1_full_reset_free_horizon)."""
    n, steps, chunk = 2048, 200000, 2000
    train, _ = eb.EARLEnvs("tabletop_manipulation", reward_type="sparse", num_envs=n, device=DEV, seed=0).get_envs()   # float32 state
    o0 = np_(train.reset())
    orc = TabletopOracle(n, steps, state_f32=False)
    orc.reset(goal_row(o0))
    rs = np.random.RandomState(123)
    obs = torch.empty((chunk, n, 12), device=DEV)
    rew = torch.empty((chunk, n), device=DEV)
    done = torch.empty((chunk, n), dtype=torch.uint8, device=DEV)
    diverged_at = np.full(n, -1, np.int64)
    attached_steps = 0
    for c in range(steps // chunk):
        # actions of a noisy mug-seeking policy driven by the CHECKER's state, so that the fist keeps hovering around the
        # 0.4 attach radius instead of random-walking away from the mug (1.5 % attached under uniform actions)
        acts = np.empty((chunk, n, 3), np.float32)
        ref_att, ref_rew = np.empty((chunk, n), np.float32), np.empty((chunk, n))
        for t in range(chunk):
            to_mug = orc.qpos[:, 2:4] - orc.qpos[:, 0:2]
            to_mug /= np.maximum(np.linalg.norm(to_mug, axis=1, keepdims=True), 1e-9)
            a = rs.uniform(-1, 1, (n, 3))
            a[:, :2] += 0.35 * to_mug
            acts[t] = a.astype(np.float32)
            o2, r2, _, _ = orc.step(acts[t])
            ref_att[t], ref_rew[t] = o2[:, 4], r2
        train.rollout_into(torch.from_numpy(acts).to(DEV), chunk, obs, rew, done)
        bad = (np_(obs[:, :, 4]) != ref_att) | (np_(rew).astype(np.float64) != ref_rew)       # attached flag, sparse reward
        first_bad = np.where(bad.any(0), bad.argmax(0) + c * chunk, -1)
        new = (first_bad >= 0) & (diverged_at < 0)
        diverged_at[new] = first_bad[new]
        attached_steps += int((ref_att == 0).sum())
    same = diverged_at < 0
    err = np.abs(train.get_state()["qpos"][same] - orc.qpos[same]).max() if same.any() else 0.0
    frac = 1.0 - same.mean()
    first = int(diverged_at[~same].min()) if (~same).any() else -1
    print(f"fp32 state vs fp64 reference, {n} envs x {steps} steps: {100 * frac:.2f} % of the envs diverge in their attach / reward "
          f"sequence (first at step {first}); max |dqpos| of the others {err:.2e}; attached env-steps {attached_steps}")
    assert attached_steps > 0.05 * n * steps                      # the decisions were exercised all along
    assert err < 1e-4                                             # north_star's one-step bar holds over the whole horizon for those
    assert frac < 0.5, frac                                       # reported, not hidden: see the printed line / DESIGN.md 3


# ---------------------------------------------------------------------------------------- round 2: kernel variants, host path

@pytest.mark.parametrize("n", [255, 4099, 70001, 3 * 2**20 + 4099])
def test_selected_step_kernels_vs_oracle(n):
    """The step kernel the library selects for the batch size -- the persistent LSU kernel up to 3M envs, the one-tile-per-CTA
    kernel above (3 * 2**20 + 4099 envs: a ragged last tile of 3 envs) -- against the oracle: ragged batches, attach / drag /
    clip, horizon `done`, host path included -- bit-exact."""
    steps, horizon = 24, 17
    env = make(n, horizon, seed=n)
    orc = TabletopOracle(n, horizon, state_f32=True)
    orc.reset(goal_row(np_(env.reset())))
    q = np.tile([0.0, 0.0, 2.5, 0.0], (n, 1))
    q[::2, 0] = 2.3
    q = q.astype(np.float32).astype(np.float64)  # representable in the fp32 state
    env.set_state(qpos=q)
    orc.qpos[:] = q
    acts = actions(n, steps, seed=7 + n, grip_bias=0.3)
    for t in range(steps):
        if t % 4 == 3:
            ob, rw, dn, info = env.step(acts[t])                      # host path drives the same kernel per chunk
            ob, rw, dn, sc = ob, rw, dn, info["success"]
        else:
            ob, rw, dn, info = env.step(torch.from_numpy(acts[t]).to(DEV))
            ob, rw, dn, sc = np_(ob), np_(rw), np_(dn), np_(info["success"])
        o2, r2, d2, s2 = orc.step(acts[t])
        assert np.array_equal(ob, o2), t
        assert np.array_equal(rw.astype(np.float64), r2) and np.array_equal(dn, d2.astype(bool)) and np.array_equal(sc, s2.astype(bool)), t
    assert (orc.attached != 0).any()


@pytest.mark.parametrize("mode", ["lifelong", "auto_reset"])
def test_chunked_host_path_reads_its_own_goal_stream(mode):
    """ADVICE r1 (medium): a chunked host step used the chunk's end as the row stride of goal_stream[R, N], so every chunk but
    the last read other envs' draws once a goal was drawn inside the step (lifelong swap, auto-reset).  Host path with 4
    chunks == device path, with goals actually changing."""
    n, steps = 4 * 2**18 + 2051, 40                                     # one chunk per 256k envs: 4 chunks
    if mode == "lifelong":
        kw = dict(setup_as_lifelong_learning=True, goal_change_frequency=7, train_horizon=10**6)
    else:
        kw = dict(auto_reset=True, train_horizon=9)
    mk = lambda: eb.EARLEnvs("tabletop_manipulation", reward_type="sparse", num_envs=n, device=DEV, seed=3, **kw).get_envs()  # noqa: E731
    a, b = mk(), mk()
    a, b = (a, b) if mode == "lifelong" else (a[0], b[0])
    oa, ob_ = np_(a.reset()), np_(b.reset())
    assert np.array_equal(oa, ob_)
    acts = actions(n, steps, seed=21, grip_bias=0.2)
    goals = set()
    launches = b.launch_count
    for t in range(steps):
        o, r, d, _ = a.step(torch.from_numpy(acts[t]).to(DEV))
        ho, hr, hd, _ = b.step(acts[t])
        assert np.array_equal(ho, np_(o)) and np.array_equal(hr, np_(r)) and np.array_equal(hd, np_(d)), t
        goals |= set(map(tuple, np.unique(ho[:, 8:10], axis=0)))
    assert b.launch_count - launches == 4 * steps                       # one step kernel per chunk: the batch ran in 4 chunks
    assert len(goals) == 4                                              # all four goals were drawn along the way


def test_host_path_outputs_do_not_alias_across_consecutive_steps():
    """ADVICE r1 (medium): `next_obs, r, d, _ = env.step(a); ...; obs = next_obs` must not see `obs` change under its feet:
    the arrays a numpy step returns stay valid during the next step (two alternating pinned sets)."""
    n = 1000
    env = make(n, 50)
    env.reset()
    acts = actions(n, 6, seed=4)
    obs, _, _, _ = env.step(acts[0])
    keep = obs.copy()
    nxt, _, _, _ = env.step(acts[1])
    assert not np.shares_memory(obs, nxt)
    assert np.array_equal(obs, keep) and not np.array_equal(obs, nxt)
    host = make(n, 50, host_io=True)
    assert isinstance(host.reset(), np.ndarray)                          # numpy-driven env: numpy out of reset() as well


def test_host_step_is_ordered_after_a_reset_on_the_callers_stream():
    """ADVICE r1 (medium): the host step runs on the handle's private non-blocking streams; a reset queued on torch's current
    stream right before it must be seen.  A long-running kernel is queued first so that an unordered step would win the race."""
    n = 1 << 18
    env, ref = make(n, 10**6), make(n, 10**6)
    acts = actions(n, 3, seed=9, grip_bias=0.5)
    for e in (env, ref):
        e.reset()
        for t in range(2):
            e.step(torch.from_numpy(acts[t]).to(DEV))
    big = torch.empty(1 << 28, device=DEV)
    for _ in range(4):
        big.normal_()                                                   # ~ms of work on the current stream ...
    env.reset()                                                          # ... then the reset, not yet executed when step() is called
    ho, hr, hd, _ = env.step(acts[2])
    ref.reset()
    torch.cuda.synchronize()
    o, r, d, _ = ref.step(torch.from_numpy(acts[2]).to(DEV))
    assert np.array_equal(ho, np_(o)) and np.array_equal(hd, np_(d))


def test_wide_init_resets_do_not_depend_on_the_sharding():
    """ADVICE r1 (low): with `wide_init_distr` every rank used to draw its initial states from its own copy of the legacy
    numpy stream, so all shards started identically and differed from the single-GPU run.  Two shards of a 600-env job ==
    the unsharded job."""
    n = 600
    whole = TabletopManipulation(num_envs=n, device=DEV, wide_init_distr=True, reward_type="sparse", seed=5)
    a = TabletopManipulation(num_envs=n // 2, device=DEV, wide_init_distr=True, reward_type="sparse", seed=5, env_offset=0, total_envs=n)
    b = TabletopManipulation(num_envs=n // 2, device=DEV, wide_init_distr=True, reward_type="sparse", seed=5, env_offset=n // 2, total_envs=n)
    ow, oa, ob = np_(whole.reset()), np_(a.reset()), np_(b.reset())
    assert np.array_equal(ow, np.concatenate([oa, ob]))
    assert not np.array_equal(oa[:, :4], ob[:, :4])


def test_lifelong_goal_stream_covers_the_horizon():
    """ADVICE r1 (low): the default lifelong tabletop run takes 50000 / 400 = 125 goal draws per env; a 64-row ring would wrap
    silently into a periodic sequence.  The ring is sized from the configuration."""
    env = eb.EARLEnvs("tabletop_manipulation", reward_type="sparse", setup_as_lifelong_learning=True, num_envs=8, device=DEV).get_envs()
    env.reset()
    base = env.env.env if hasattr(env.env, "env") else env.env
    assert base._goal_stream.shape[0] >= 127


@pytest.mark.parametrize("n", [2051, 3 * 2**20 + 2051])               # the latter: 12 chunks of the copy pipeline
def test_zero_copy_host_step_equals_the_copy_pipeline_and_the_device_path(monkeypatch, n):
    """EARL_TT_HOST_ZEROCOPY=1: the one-tile-per-CTA step kernel reads the pinned host actions and writes the pinned host
    outputs itself (no staging copies).  Same observations, rewards, done / success flags and state as the chunked copy
    pipeline and as the device-resident step, bit for bit, on a ragged and on a multi-chunk batch."""
    steps = 12
    acts = actions(n, steps, seed=31, grip_bias=0.3)
    monkeypatch.setenv("EARL_TT_HOST_ZEROCOPY", "1")
    z = make(n, 7)
    monkeypatch.setenv("EARL_TT_HOST_ZEROCOPY", "0")
    c, d = make(n, 7), make(n, 7)
    for e in (z, c, d):
        e.reset()
    for t in range(steps):
        zo, zr, zd, zi = z.step(acts[t])
        co, cr, cd, ci = c.step(acts[t])
        do, dr, dd, di = d.step(torch.from_numpy(acts[t]).to(DEV))
        assert isinstance(zo, np.ndarray)
        assert np.array_equal(zo, co) and np.array_equal(zr, cr) and np.array_equal(zd, cd) and np.array_equal(zi["success"], ci["success"]), t
        assert np.array_equal(zo, np_(do)) and np.array_equal(zr, np_(dr)) and np.array_equal(zd, np_(dd)), t
    assert zd.all()                                                      # the horizon (7) was crossed inside the run
    sz, sd = z.env.get_state(), d.env.get_state()
    for k in sz:
        assert np.array_equal(np.asarray(sz[k]), np.asarray(sd[k])), k
