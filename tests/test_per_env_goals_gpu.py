"""Per-env goals set on the device (`per_env_goals=True`: set_goals / get_goals) for tabletop_manipulation, sawyer_door and
sawyer_peg: parity with the goal-table path, immediate effect, masks, scale beyond the goal-table limits, the reference's
reset / auto-reset / lifelong semantics, errors, and launch counts."""
import numpy as np
import pytest
import torch

import earl_benchmark_b200 as eb
from earl_benchmark_b200.envs import sawyer_door, sawyer_peg
from earl_benchmark_b200.envs.tabletop_manipulation import TabletopManipulation
from earl_benchmark_b200.wrappers.lifelong_wrapper import LifelongWrapper
from earl_benchmark_b200.wrappers.persistent_state_wrapper import PersistentStateWrapper

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NEVER = 1 << 40


def rand_actions(shape, seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return torch.rand(shape, generator=g, device=DEV) * 2 - 1


def rand_mask(n, seed):
    return torch.from_numpy(np.random.RandomState(seed).rand(n) < 0.5).to(DEV)


def table(env, rows):
    return torch.from_numpy(np.stack([env._goal_table[r] for r in np.asarray(rows)])).to(DEV)   # float64


def goal_slice(env):
    return slice(6, 12) if isinstance(env, TabletopManipulation) else slice(7, 14)


def same(a, b):
    return torch.equal(torch.as_tensor(a), torch.as_tensor(b))


# ------------------------------------------------------------------------------------------------ 1. parity (tabletop)
@pytest.mark.parametrize("state_dtype", ["float32", "float64"])
@pytest.mark.parametrize("reward_type", ["sparse", "dense"])
@pytest.mark.parametrize("path", ["device", "rollout", "host"])
def test_tabletop_set_goals_matches_goal_table_rows(state_dtype, reward_type, path):
    if path != "device" and (state_dtype, reward_type) != ("float32", "sparse"):
        pytest.skip("the rollout and host paths run once, on the headline configuration")
    n, steps = 4096, 200
    kw = dict(reward_type=reward_type, state_dtype=state_dtype, num_envs=n, device=DEV, seed=7)
    ref, env = TabletopManipulation(**kw), TabletopManipulation(per_env_goals=True, **kw)
    rs = np.random.RandomState(1)
    rows = rs.randint(0, 5, n)
    ref.reset(goal_rows=rows)
    env.reset(goal_rows=np.zeros(n, np.int32))
    assert same(env.set_goals(table(env, rows)), ref.get_obs())
    rows2, mask = rs.randint(0, 5, n), rand_mask(n, 2)
    acts = rand_actions((steps, n, 3), 3)

    def change_goals():   # second goal change, float32 input, half the envs
        ref.reset_goal(np.stack([ref._goal_table[r] for r in rows2]), mask=mask)
        assert same(env.set_goals(table(env, rows2).float(), mask=mask), ref.get_obs())

    if path == "rollout":
        for half in range(2):
            outs = []
            for e in (ref, env):
                o = torch.empty((steps // 2, n, 12), device=DEV)
                r = torch.empty((steps // 2, n), device=DEV)
                d = torch.empty((steps // 2, n), dtype=torch.uint8, device=DEV)
                s = torch.empty((steps // 2, n), dtype=torch.uint8, device=DEV)
                e.rollout_into(acts[half * steps // 2:(half + 1) * steps // 2].contiguous(), steps // 2, o, r, d, s)
                outs.append((o, r, d, s))
            for a, b in zip(*outs):
                assert same(a, b), half
            if half == 0:
                change_goals()
        return
    hits = 0
    for t in range(steps):
        if t == steps // 2:
            change_goals()
        a = acts[t] if path == "device" else acts[t].cpu().numpy()
        o1, r1, d1, i1 = ref.step(a)
        o2, r2, d2, i2 = env.step(a)
        assert same(o1, o2) and same(r1, r2) and same(d1, d2) and same(i1["success"], i2["success"]), t
        hits += int(torch.as_tensor(i2["success"]).sum())
    assert hits > 0


# ------------------------------------------------------------------------------------------------ 1. parity (Sawyer)
SAWYER = {
    "door-sparse": (sawyer_door.SawyerDoorV2, dict(reward_type="sparse")),
    "door-dense": (sawyer_door.SawyerDoorV2, dict(reward_type="dense")),
    "peg-sparse": (sawyer_peg.SawyerPegV2, dict(reward_type="sparse")),
    "peg-dense": (sawyer_peg.SawyerPegV2, dict(reward_type="dense")),
}


def sawyer_reset(env, mask, rs_seed):
    """a reset with explicit draws (the goal row then comes from reset_goal: peg's own draw always assigns row 0)"""
    rs = np.random.RandomState(rs_seed)
    if isinstance(env, sawyer_peg.SawyerPegV2):
        pos = np.tile([0.0, 0.6, 0.02], (env.num_envs, 1)) + np.c_[rs.uniform(-0.05, 0.05, (env.num_envs, 2)), np.zeros(env.num_envs)]
        return env.reset(mask=mask, peg_pos=pos)
    return env.reset(mask=mask, door_angle=rs.uniform(-np.pi / 3, -np.pi / 3 + np.pi / 20, env.num_envs))


@pytest.mark.parametrize("name", list(SAWYER))
def test_sawyer_set_goals_matches_goal_table_rows(name):
    cls, opts = SAWYER[name]
    n, steps = 512, 200
    ref, env = cls(num_envs=n, device=DEV, seed=5, **opts), cls(num_envs=n, device=DEV, seed=5, per_env_goals=True, **opts)
    assert same(sawyer_reset(ref, None, 0), sawyer_reset(env, None, 0))
    goals = [ref._goal_table[1], ref._goal_table[-1], ref._goal_table[0]]
    acts = rand_actions((steps, n, 4), 11)
    for t in range(steps):
        if t in (0, 1, steps // 2):   # custom goals on overlapping masks, float64 then float32 input
            k = (0, 1, 2)[(0, 1, steps // 2).index(t)]
            mask = rand_mask(n, 20 + k)
            ref.reset_goal(goals[k])
            o1 = sawyer_reset(ref, mask, 30 + k)
            sawyer_reset(env, mask, 30 + k)
            g = torch.from_numpy(goals[k]).to(DEV)
            o2 = env.set_goals(g if k != 2 else g.float(), mask=mask)
            assert same(o1, o2), t
        o1, r1, d1, i1 = ref.step(acts[t])
        o2, r2, d2, i2 = env.step(acts[t])
        assert same(o1, o2) and same(r1, r2) and same(d1, d2) and same(i1["success"], i2["success"]), t


# ------------------------------------------------------------------------------------------------ 2. immediate effect, masks
def near_goals(env, obs, seed, spread):
    """random goals whose target lies within `spread` of the object, so that the next step succeeds for some envs only"""
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    n = env.num_envs
    if isinstance(env, TabletopManipulation):
        goals = torch.rand((n, 6), generator=g, device=DEV, dtype=torch.float64) * 5 - 2.5
        goals[:, 0:4] = obs[:, 0:4].double() + (torch.rand((n, 4), generator=g, device=DEV, dtype=torch.float64) * 2 - 1) * spread
    else:
        goals = torch.rand((n, 7), generator=g, device=DEV, dtype=torch.float64) * 0.4
        goals[:, 4:7] = obs[:, 4:7].double() + (torch.rand((n, 3), generator=g, device=DEV, dtype=torch.float64) * 2 - 1) * spread
    return goals


def check_success(env, obs, success, reward):
    """success / reward of a step against the cold-path formulas on that step's observation"""
    if isinstance(env, TabletopManipulation):
        assert same(success, env.is_successful(obs)) and same(reward, env.compute_reward(obs))
        return
    o = obs.double()
    dist = torch.linalg.norm(o[:, 4:7] - o[:, 11:14], dim=1)
    want = dist <= env.SUCCESS_RADIUS
    # the kernel takes the fp32 norm: only a distance within rounding of the radius may decide differently
    bad = (success != want) & ((dist - env.SUCCESS_RADIUS).abs() > 1e-6)
    assert not bool(bad.any())
    if env._reward_type == "sparse":
        assert same(reward, success.float())
    else:
        assert float((reward - env.compute_reward(obs)).abs().max()) < 2e-4


@pytest.mark.parametrize("name", ["tabletop-sparse", "tabletop-dense", "door-sparse", "door-dense", "peg-sparse"])
def test_set_goals_takes_effect_at_once_and_respects_the_mask(name):
    if name.startswith("tabletop"):
        n, spread = 4096, 0.15
        env = TabletopManipulation(reward_type=name.split("-")[1], num_envs=n, device=DEV, seed=2, per_env_goals=True)
        adim = 3
    else:
        cls, opts = SAWYER[name]
        n, spread = 1024, 0.04
        env = cls(num_envs=n, device=DEV, seed=2, per_env_goals=True, **opts)
        adim = 4
    env.reset()
    acts = rand_actions((12, n, adim), 4)
    for t in range(12):
        obs, _, _, _ = env.step(acts[t])
        if t % 4 != 3:
            continue
        before = env.get_obs().clone()
        if isinstance(env, TabletopManipulation):
            assert same(before, obs)
        goals, mask = near_goals(env, before, 50 + t, spread), rand_mask(n, 60 + t)
        out = env.set_goals(goals, mask=mask)
        sl = goal_slice(env)
        m = mask.bool()
        assert same(out[m][:, sl], goals[m].float())
        assert same(out[~m], before[~m])
        assert same(env.get_goals(), out[:, sl])
        assert same(env.get_obs(), out)
        nobs, rew, _, info = env.step(acts[(t + 1) % 12])
        assert same(nobs[:, sl], out[:, sl])
        check_success(env, nobs, info["success"], rew)
        s = info["success"][m]
        assert 0 < int(s.sum()) < int(m.sum()), name
        obs = nobs


def test_host_io_env_takes_numpy_goals_and_returns_numpy():
    n = 64
    env = TabletopManipulation(reward_type="sparse", num_envs=n, device=DEV, per_env_goals=True, host_io=True)
    env.reset()
    goals = np.random.RandomState(0).uniform(-2, 2, (n, 6))
    mask = np.arange(n) % 2 == 0
    out = env.set_goals(goals, mask=mask)
    assert isinstance(out, np.ndarray) and np.array_equal(out[mask, 6:12], goals[mask].astype(np.float32))
    assert np.array_equal(env.get_goals().cpu().numpy()[mask], goals[mask].astype(np.float32))
    door = sawyer_door.SawyerDoorV2(num_envs=8, device=DEV, per_env_goals=True, host_io=True)
    door.reset()
    out = door.set_goals(sawyer_door.goal_states[0] + 0.01)
    assert isinstance(out, np.ndarray) and np.array_equal(out[:, 7:14], np.tile((sawyer_door.goal_states[0] + 0.01).astype(np.float32), (8, 1)))


# ------------------------------------------------------------------------------------------------ 3. scale
@pytest.mark.parametrize("name,n", [("tabletop", 65536), ("door", 4096), ("peg", 4096)])
def test_every_env_gets_its_own_goal_every_step(name, n):
    """far beyond the 256 (tabletop) and 32 (Sawyer) goal-table rows: a new random goal per env and step"""
    if name == "tabletop":
        env, adim, spread = TabletopManipulation(reward_type="sparse", num_envs=n, device=DEV, seed=1, per_env_goals=True), 3, 0.15
    else:
        cls = sawyer_door.SawyerDoorV2 if name == "door" else sawyer_peg.SawyerPegV2
        env, adim, spread = cls(reward_type="sparse", num_envs=n, device=DEV, seed=1, per_env_goals=True), 4, 0.04
    obs = env.reset()
    sl = goal_slice(env)
    hits = 0
    for t in range(100):
        goals = near_goals(env, obs, 1000 + t, spread)
        mask = rand_mask(n, t) if t % 3 == 2 else None
        want = env.get_goals().clone()
        if mask is None:
            want = goals.float()
        else:
            want[mask] = goals[mask].float()
        out = env.set_goals(goals, mask=mask)
        assert same(out[:, sl], want)
        obs, rew, _, info = env.step(rand_actions((n, adim), 2000 + t))
        assert same(obs[:, sl], want) and same(env.get_goals(), want)
        check_success(env, obs, info["success"], rew)
        hits += int(info["success"].sum())
    assert hits > 0


# ------------------------------------------------------------------------------------------------ 4. reference semantics
def custom_goals(env, seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return torch.rand((env.num_envs, 6 if isinstance(env, TabletopManipulation) else 7), generator=g, device=DEV, dtype=torch.float64) + 5.0


def task_goals(env):
    """the goal-table row each env was last assigned, float32"""
    if isinstance(env, TabletopManipulation):
        rows = env.get_state()["goal_row"]
    else:
        rows = env._goal_rows.cpu().numpy()
    return table(env, rows).float()


def check_event(env, obs, touched, custom):
    """envs in `touched` pursue the task's goal again, the others keep their custom goal; obs carries what get_goals says"""
    got = env.get_goals()
    assert same(got[touched], task_goals(env)[touched])
    assert same(got[~touched], custom.float()[~touched])
    assert same(obs[:, goal_slice(env)], got)


@pytest.mark.parametrize("name", ["tabletop", "door"])
def test_masked_reset_restores_the_task_goal(name):
    n = 1024
    env = (TabletopManipulation(num_envs=n, device=DEV, per_env_goals=True) if name == "tabletop"
           else sawyer_door.SawyerDoorV2(num_envs=n, device=DEV, per_env_goals=True))
    env.reset()
    custom = custom_goals(env, 1)
    env.set_goals(custom)
    mask = rand_mask(n, 3)
    obs = env.reset(mask=mask)
    check_event(env, obs, mask, custom)
    if name == "tabletop":   # reset_goal(None) assigns the next stream row; get_next_goal() changes nobody's goal
        env.set_goals(custom)
        env.reset_goal(mask=mask)
        check_event(env, env.get_obs(), mask, custom)
        before = env.get_goals().clone()
        env.get_next_goal()
        assert same(env.get_goals(), before)
        assert np.array_equal(env.goal, before.cpu().numpy().astype(np.float64))


@pytest.mark.parametrize("name", ["tabletop", "door"])
@pytest.mark.parametrize("event", ["auto_reset", "lifelong"])
def test_auto_reset_and_lifelong_swap_restore_the_task_goal(name, event):
    n, period = 1024, 4
    kw = dict(num_envs=n, device=DEV, per_env_goals=True, auto_reset=(event == "auto_reset"))
    base = TabletopManipulation(**kw) if name == "tabletop" else sawyer_door.SawyerDoorV2(**kw)
    env = PersistentStateWrapper(base, period if event == "auto_reset" else NEVER)
    if event == "lifelong":
        env = LifelongWrapper(env, period)
    adim = 3 if name == "tabletop" else 4
    env.reset()
    for t in range(2):
        env.step(rand_actions((n, adim), t))
    mask = rand_mask(n, 5)
    env.reset(mask=mask)       # these envs restart their horizon / goal-change count: the event skips them below
    custom = custom_goals(base, 6)
    base.set_goals(custom)
    obs, _, done, _ = env.step(rand_actions((n, adim), 10))
    assert same(obs[:, goal_slice(base)], custom.float())
    obs, _, done, _ = env.step(rand_actions((n, adim), 11))
    if event == "auto_reset":
        assert same(done, ~mask)
    check_event(base, obs, ~mask, custom)


# ------------------------------------------------------------------------------------------------ 5. errors
def test_errors():
    plain = TabletopManipulation(num_envs=8, device=DEV)
    plain.reset()
    with pytest.raises(RuntimeError):
        plain.set_goals(torch.zeros(6, device=DEV))
    with pytest.raises(RuntimeError):
        plain.get_goals()
    door_plain = sawyer_door.SawyerDoorV2(num_envs=8, device=DEV)
    with pytest.raises(RuntimeError):
        door_plain.set_goals(torch.zeros(7, device=DEV))
    for env, width in ((TabletopManipulation(num_envs=8, device=DEV, per_env_goals=True), 6),
                       (sawyer_door.SawyerDoorV2(num_envs=8, device=DEV, per_env_goals=True), 7),
                       (sawyer_peg.SawyerPegV2(num_envs=8, device=DEV, per_env_goals=True), 7)):
        env.reset()
        with pytest.raises(ValueError):
            env.set_goals(torch.zeros((8, width + 1), device=DEV))
        with pytest.raises(ValueError):
            env.set_goals(torch.zeros((9, width), device=DEV))
        with pytest.raises(TypeError):
            env.set_goals(torch.zeros((8, width), dtype=torch.int32, device=DEV))
        with pytest.raises(TypeError):
            env.set_goals(torch.zeros((8, width)))                     # CPU input on a device env
        with pytest.raises(ValueError):
            env.set_goals(torch.zeros((8, width), device=DEV), mask=torch.ones(7, dtype=torch.bool, device=DEV))
    with pytest.raises(NotImplementedError):
        eb.EARLEnvs("kitchen", num_envs=4, per_env_goals=True)


def test_earl_envs_passes_the_flag_to_train_and_eval_envs():
    for name in ("tabletop_manipulation", "sawyer_door", "sawyer_peg"):
        tr, ev = eb.EARLEnvs(name, num_envs=16, per_env_goals=True).get_envs()
        for e in (tr, ev):
            e.reset()
            assert e.get_goals().shape == (16, 6 if name == "tabletop_manipulation" else 7)
    tr = eb.EARLEnvs("tabletop_manipulation", num_envs=16, setup_as_lifelong_learning=True, per_env_goals=True).get_envs()
    tr.reset()
    assert tr.get_goals().shape == (16, 6)
    tr, _ = eb.EARLEnvs("sawyer_door", num_envs=16).get_envs()
    with pytest.raises(RuntimeError):
        tr.get_goals()


# ------------------------------------------------------------------------------------------------ 6. launches, kernels
@pytest.mark.parametrize("name", ["tabletop", "door", "peg"])
def test_set_goals_is_one_launch_without_synchronisation(name):
    n = 256
    if name == "tabletop":
        env, width, get_launches = TabletopManipulation(num_envs=n, device=DEV, per_env_goals=True), 6, 0
    else:
        cls = sawyer_door.SawyerDoorV2 if name == "door" else sawyer_peg.SawyerPegV2
        env, width, get_launches = cls(num_envs=n, device=DEV, per_env_goals=True), 7, 1
    env.reset()
    goals, mask = torch.rand((n, width), device=DEV, dtype=torch.float64), rand_mask(n, 1)
    torch.cuda.synchronize()
    before = env.launch_count
    torch.cuda.set_sync_debug_mode("error")   # any host synchronisation torch would make raises
    try:
        env.set_goals(goals, mask=mask)
        env.set_goals(goals[0].float())
        after_set = env.launch_count
        env.get_goals()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert after_set - before == 2
    assert env.launch_count - after_set == get_launches


def step_kernel_names(env, action):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        env.step(action)
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if "tabletop_step" in e.name]


@pytest.mark.parametrize("kw", [dict(reward_type="sparse"), dict(reward_type="dense"), dict(reward_type="dense", state_dtype="float64")])
def test_default_handles_keep_their_step_kernel(kw):
    n = 4096
    a = rand_actions((n, 3), 0)
    plain = TabletopManipulation(num_envs=n, device=DEV, **kw)
    goals = TabletopManipulation(num_envs=n, device=DEV, per_env_goals=True, **kw)
    plain.reset()
    goals.reset()
    fast = kw["reward_type"] == "sparse"
    for env, want in ((plain, "true" if fast else "false"), (goals, "false")):
        names = step_kernel_names(env, a)
        per_env = "true" if env is goals else "false"
        assert names and all(f"tabletop_step_kernel<{'true' if 'float64' in kw.values() else 'false'}, {want}, 1, {per_env}>" in k
                             for k in names), names
