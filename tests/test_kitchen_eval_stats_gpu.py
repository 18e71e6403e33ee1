"""Kitchen evaluation statistics on the device (Kitchen(eval_stats=True), earl_mjk_eval_stats): the [4] tensor equals a host
accumulation of the rewards and successes the steps return, any reset clears an env's statistics, and the flag changes
nothing else the kitchen computes."""
import numpy as np
import pytest
import torch

import earl_benchmark_b200 as eb
from earl_benchmark_b200 import _lib
from earl_benchmark_b200.distributed import all_reduce_eval_stats
from earl_benchmark_b200.envs import kitchen
from earl_benchmark_b200.wrappers.persistent_state_wrapper import PersistentStateWrapper

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOAL_OBJ = kitchen.goal_states[0][9:]
SLIDE = kitchen.component_to_state_idx['slide_cabinet'][0]


class HostStats:
    """Per env, in step order: the returned rewards summed and the returned successes (any step / last step)."""

    def __init__(self, n):
        self.ret, self.any, self.last = np.zeros(n), np.zeros(n, bool), np.zeros(n, bool)

    def step(self, reward, success):
        reward = reward.cpu().numpy() if isinstance(reward, torch.Tensor) else np.asarray(reward)
        success = success.cpu().numpy() if isinstance(success, torch.Tensor) else np.asarray(success)
        self.ret += reward
        self.last = success.astype(bool).copy()
        self.any |= self.last

    def reset(self, mask=None):
        m = slice(None) if mask is None else np.asarray(mask.cpu() if isinstance(mask, torch.Tensor) else mask, bool)
        self.ret[m], self.any[m], self.last[m] = 0.0, False, False

    def check(self, got, where=""):
        got = got.cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
        assert got.dtype == np.float64 and got.shape == (4,)
        want = [self.last.sum(), self.any.sum(), len(self.ret)]
        assert got[1:].tolist() == want, (where, got, want)
        # the per-env returns are the same bits; only the order of the sum over envs differs from numpy's
        assert abs(got[0] - self.ret.sum()) <= 1e-12 * max(np.abs(self.ret).sum(), 1e-300), (where, got[0], self.ret.sum())


def make(n, seed=3, horizon=1 << 40, **kw):
    return PersistentStateWrapper(kitchen.Kitchen(num_envs=n, device=DEV, seed=seed, **kw), horizon)


def put_objects_at_goal(envs, ids, slide_offset=0.0):
    """Objects of envs `ids` at the goal state (success), the slide cabinet moved by `slide_offset`; same state on every
    handle in `envs` (which must hold the same state)."""
    st = envs[0].get_state()
    q = st["qpos"].copy()
    q[ids, 9:] = GOAL_OBJ
    q[ids, SLIDE] += slide_offset
    for e in envs:
        e.set_state(qpos=q)


def actions(n, steps, seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return torch.rand((steps, n, 9), generator=g, device=DEV) * 2 - 1


def test_statistics_follow_the_returned_rewards_and_successes():
    n, horizon, steps = 64, 6, 14
    env = make(n, 5, horizon, eval_stats=True)
    ref = HostStats(n)
    env.reset(config_index=np.arange(n) % 6)
    ref.check(env.eval_stats(), "after the first reset")
    # envs 40-47 at the goal (successful), 48-63 with the slide cabinet 0.3 off it: the observation noise flips their success
    put_objects_at_goal([env], np.arange(40, 48))
    put_objects_at_goal([env], np.arange(48, 64), slide_offset=0.3)
    acts = actions(n, steps, 6)
    masks = {2: np.arange(n) < 16, 5: (np.arange(n) >= 8) & (np.arange(n) < 40), 9: np.arange(n) % 2 == 1}
    host_steps = (3, 10)
    any_not_last = False
    for t in range(steps):
        if t in host_steps:
            o, r, d, info = env.step(acts[t].cpu().numpy())
            assert isinstance(r, np.ndarray)
        else:
            o, r, d, info = env.step(acts[t])
        ref.step(r, info["success"])
        ref.check(env.eval_stats(), f"step {t}")
        any_not_last |= bool((ref.any & ~ref.last).any())
        if t in masks:
            env.reset(mask=masks[t])
            ref.reset(masks[t])
            ref.check(env.eval_stats(), f"masked reset after step {t}")
    assert env.total_steps == steps and bool(d[torch.from_numpy(~masks[9]).to(DEV)].all())   # past the horizon, still counting
    assert ref.last.sum() > 0 and any_not_last                        # both success bits were exercised
    a, b = env.eval_stats(), env.eval_stats()
    assert torch.equal(a, b)
    env.reset()
    assert env.eval_stats().tolist() == [0.0, 0.0, 0.0, float(n)]


def scripted_reach(env, n, steps, gen_seed, ref=None):
    """test_redo_scheduling_does_not_change_the_kitchen_physics's policy: every arm driven into the slide-cabinet handle."""
    k = kitchen.REWARD_SITES.index("slide_site")
    gen = torch.Generator(device=DEV)
    gen.manual_seed(gen_seed)
    out = []
    for t in range(steps):
        st = env.get_state()
        d = torch.from_numpy(st["site_xpos"][:, k] - st["mocap_pos"]).to(DEV, torch.float32)
        u = torch.zeros((n, 9), device=DEV)
        u[:, :3] = torch.clamp(d * 10, -1, 1) * 0.5
        u += 0.1 * (torch.rand((n, 9), generator=gen, device=DEV) * 2 - 1)
        ob, r, dn, info = env.step(u)
        out.append((ob.clone(), r.clone(), dn.clone(), info["success"].clone()))
        if ref is not None:
            ref.step(r, info["success"])
    return out


def test_the_flag_changes_nothing_else():
    n, steps = 592, 70

    def run(flag):
        env = make(n, 4, eval_stats=flag)
        env.seed(4)
        env.reset()
        put_objects_at_goal([env], np.arange(0, n, 7))
        ref = HostStats(n)
        out = scripted_reach(env, n, steps, 8, ref)
        return env, out, ref

    e0, out0, _ = run(False)
    e1, out1, ref = run(True)
    w0, w1 = e0.work_counters(), e1.work_counters()
    if w0["redone_states"] == 0:
        pytest.skip("the scripted reach no longer outgrows the primary capacity set")
    assert w0 == w1
    for t, (a, b) in enumerate(zip(out0, out1)):
        for x, y in zip(a, b):
            assert torch.equal(x, y), t
    s0, s1 = e0.get_state(), e1.get_state()
    for key in s0:
        assert np.array_equal(s0[key], s1[key]), key
    c0, c1 = e0.env._counters(), e1.env._counters()
    assert c0[0] == c1[0] and torch.equal(c0[1], c1[1]) and torch.equal(c0[2], c1[2])
    ref.check(e1.eval_stats())
    assert ref.any.sum() > 0
    with pytest.raises(_lib.EarlError) as ei:
        e0.eval_stats()
    assert ei.value.code == -1 and "EARL_FLAG_EVAL_STATS" in str(ei.value)


def test_statistics_without_the_redo_pass(monkeypatch):
    monkeypatch.setenv("EARL_MJ_REDO", "0")
    n = 296
    env = make(n, 4, eval_stats=True)
    env.seed(4)
    env.reset()
    ref = HostStats(n)
    scripted_reach(env, n, 40, 9, ref)
    assert env.work_counters()["redone_states"] == 0
    ref.check(env.eval_stats())


def test_a_failed_step_adds_nothing_and_is_not_a_success():
    n, bad = 4, 1
    env = make(n, 2, eval_stats=True)
    env.seed(2)
    env.reset(config_index=np.arange(n))
    put_objects_at_goal([env], np.arange(n))
    ref = HostStats(n)
    a = np.random.RandomState(0).uniform(-1, 1, (n, 9)).astype(np.float32)
    _, r, _, info = env.step(torch.from_numpy(a).cuda())
    ref.step(r, info["success"])
    assert bool(info["success"].all())
    ref.check(env.eval_stats())
    before = env.eval_stats().cpu().numpy()
    st = env.get_state()
    st["qvel"][bad, 2] = 3e38
    env.set_state(qvel=st["qvel"])
    _, r, _, info = env.step(torch.from_numpy(a).cuda())
    r, s = r.cpu().numpy(), info["success"].cpu().numpy()
    assert r[bad] == 0.0 and not s[bad] and s[np.arange(n) != bad].all() and env.work_counters()["bad_states"] == 1
    ref.step(r, s)
    ref.check(env.eval_stats())
    got = env.eval_stats().cpu().numpy()
    assert got[1:].tolist() == [n - 1, n, n]                          # bit 1 lost, bit 0 kept
    others = r[np.arange(n) != bad]
    assert abs(got[0] - (before[0] + others.sum())) <= 1e-12 * (abs(before[0]) + np.abs(others).sum())


@pytest.mark.parametrize("case", ["all_pairs-wrapping_stream", "microwave-staggered"])
def test_auto_reset_statistics_equal_a_manual_reset(case):
    n, seed = 48, 7
    if case.startswith("all_pairs"):
        horizon, steps, rows = 4, 4 * 4 + 1, 3
        auto = make(n, seed, horizon, task="all_pairs", auto_reset=True, reset_stream_rows=rows, eval_stats=True)
        manual = make(n, seed, horizon, task="all_pairs", eval_stats=True)
        # the manual handle resets from the same (wrapping) stream rows the auto-reset handle reads
        config = kitchen.reset_stream(seed, n, 0, n, rows, "all_pairs")[0]
        resets = 0
        oa, om = auto.reset(), manual.reset(config_index=config[0])
        early = {}
    else:
        horizon, steps, rows = 5, 3 * 5 + 1, 64
        auto = make(n, seed, horizon, task="microwave", auto_reset=True, eval_stats=True)
        manual = make(n, seed, horizon, task="microwave", eval_stats=True)
        config = None
        oa, om = auto.reset(), manual.reset()
        early = {0: np.arange(n) < 16, 1: (np.arange(n) >= 16) & (np.arange(n) < 40)}
    assert torch.equal(oa, om)
    put_objects_at_goal([auto, manual], np.arange(0, n, 3))
    put_objects_at_goal([auto, manual], np.arange(1, n, 3), slide_offset=0.3)
    acts = actions(n, steps, seed + 1)
    for t in range(steps):
        oa, ra, da, ia = auto.step(acts[t])
        om, rm, dm, im = manual.step(acts[t])
        assert torch.equal(ra, rm) and torch.equal(da, dm) and torch.equal(ia["success"], im["success"]), t
        if bool(dm.any()):
            if config is None:
                om = manual.reset(mask=dm)
            else:
                assert bool(dm.all())                                 # lockstep: aligned horizons
                resets += 1
                om = manual.reset(mask=dm, config_index=config[resets % rows])
        assert torch.equal(oa, om), t
        assert torch.equal(auto.eval_stats(), manual.eval_stats()), t
        if t in early:
            auto.reset(mask=early[t])
            manual.reset(mask=early[t])
            assert torch.equal(auto.eval_stats(), manual.eval_stats()), t
    if config is not None:
        assert resets > rows - 1                                      # the stream wrapped
    assert torch.equal(auto.num_interventions, manual.num_interventions)


def test_lifelong_goal_swap_steps():
    n, steps = 32, 9

    def run(flag):
        env = make(n, 2, eval_stats=flag)
        env.env._configure(lifelong=True, goal_change_frequency=2)
        env.reset()
        ref = HostStats(n)
        acts = actions(n, steps, 3)
        for t in range(steps):
            _, r, _, info = env.step(acts[t])
            ref.step(r, info["success"])
        return env, ref

    e0, _ = run(False)
    e1, ref = run(True)
    ref.check(e1.eval_stats())
    assert torch.equal(e0.env._counters(want_ll=True)[3], e1.env._counters(want_ll=True)[3])
    assert np.array_equal(e1.env._counters(want_ll=True)[3].cpu().numpy(), ref.ret)   # no reset: the same per-env sums


def test_loader_eval_env_and_the_all_reduce():
    n, horizon = 24, 5
    _, ev = eb.EARLEnvs("kitchen", reward_type="dense", num_envs=n, seed=3, eval_horizon=horizon, device=DEV).get_envs()
    assert ev.env._eval_stats
    ev.reset()
    put_objects_at_goal([ev], np.arange(0, n, 4))
    ref = HostStats(n)
    acts = actions(n, horizon, 12)
    for t in range(horizon):
        _, r, d, info = ev.step(acts[t])
        ref.step(r, info["success"])
    assert bool(d.all())
    stats = ev.eval_stats()
    ref.check(stats)
    m = all_reduce_eval_stats(stats)
    assert m["num_envs"] == n and m["success_rate"] == ref.last.sum() / n and m["success_any_rate"] == ref.any.sum() / n
    assert abs(m["mean_return"] - ref.ret.mean()) <= 1e-12 * np.abs(ref.ret).mean()
    _, plain = eb.EARLEnvs("kitchen", reward_type="dense", num_envs=4, eval_stats=False, device=DEV).get_envs()
    with pytest.raises(_lib.EarlError):
        plain.eval_stats()


def test_shards_sum_to_the_unsharded_handle():
    n, world, horizon = 40, 3, 6

    def eval_env(rank, size):
        return eb.EARLEnvs("kitchen", reward_type="dense", num_envs=n, seed=9, eval_horizon=horizon, device=DEV,
                           rank=rank, world_size=size).get_envs()[1]

    full = eval_env(0, 1)
    shards = [eval_env(r, world) for r in range(world)]
    full.reset()
    for s in shards:
        s.reset()
    q = full.get_state()["qpos"].copy()
    q[::5, 9:] = GOAL_OBJ
    full.set_state(qpos=q)
    for s in shards:
        lo = s.env._env_offset
        s.set_state(qpos=q[lo:lo + s.env.num_envs])
    acts = actions(n, horizon + 2, 13)
    for t in range(horizon + 2):
        full.step(acts[t])
        for s in shards:
            lo = s.env._env_offset
            s.step(acts[t, lo:lo + s.env.num_envs].contiguous())
    want = full.eval_stats().cpu().numpy()
    parts = np.stack([s.eval_stats().cpu().numpy() for s in shards])
    got = parts.sum(0)
    assert got[1:].tolist() == want[1:].tolist() and want[3] == n and want[1] > 0
    assert abs(got[0] - want[0]) <= 1e-12 * np.abs(parts[:, 0]).sum()


def test_repeated_reductions_are_bit_identical():
    n = 2500                                                          # more envs than threads: the strided sums iterate
    env = make(n, 1, eval_stats=True)
    env.reset()
    acts = actions(n, 3, 2)
    for t in range(3):
        env.step(acts[t])
    first = env.eval_stats()
    for _ in range(3):
        assert torch.equal(env.eval_stats(), first)
