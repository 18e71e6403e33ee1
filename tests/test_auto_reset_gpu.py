"""Auto-reset of the articulated-body tasks (sawyer_door, sawyer_peg, kitchen): the reset the step launches when the horizon
fires equals the user calling reset() after done, bit for bit, and handles without the flag launch what they always did."""
import numpy as np
import pytest
import torch

import earl_benchmark_b200 as eb
from earl_benchmark_b200.envs import kitchen, sawyer_door, sawyer_peg
from earl_benchmark_b200.wrappers.persistent_state_wrapper import PersistentStateWrapper

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

DOOR_PEG = {
    "door-sparse": (sawyer_door.SawyerDoorV2, dict(reward_type="sparse", eval_stats=True)),
    "door-dense": (sawyer_door.SawyerDoorV2, dict(reward_type="dense")),
    "door-reset_at_goal": (sawyer_door.SawyerDoorV2, dict(reset_at_goal=True)),
    "peg-sparse": (sawyer_peg.SawyerPegV2, dict(reward_type="sparse", eval_stats=True)),
    "peg-dense": (sawyer_peg.SawyerPegV2, dict(reward_type="dense")),
    "peg-wide_init": (sawyer_peg.SawyerPegV2, dict(wide_init=True)),
    "peg-reset_at_goal": (sawyer_peg.SawyerPegV2, dict(reset_at_goal=True)),
}
KITCHEN = {"kitchen-all_pairs": dict(task="all_pairs"), "kitchen-microwave": dict(task="microwave")}


def make(name, horizon, n, seed=3, **kw):
    if name in KITCHEN:
        env = kitchen.Kitchen(num_envs=n, device=DEV, seed=seed, **KITCHEN[name], **kw)
    else:
        cls, opts = DOOR_PEG[name]
        env = cls(num_envs=n, device=DEV, seed=seed, **opts, **kw)
    return PersistentStateWrapper(env, horizon)


def actions(name, n, steps, seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    dim = 9 if name in KITCHEN else 4
    return torch.rand((steps, n, dim), generator=g, device=DEV) * 2 - 1


def state_arrays(env):
    return {k: v for k, v in env.get_state().items()}


def compare_auto_and_manual(name, n, horizon, steps, seed=3, acts=None, **kw):
    auto, manual = make(name, horizon, n, seed, auto_reset=True, **kw), make(name, horizon, n, seed, **kw)
    oa, om = auto.reset(), manual.reset()
    assert torch.equal(oa, om)
    acts = actions(name, n, steps, seed + 1) if acts is None else acts
    for t in range(steps):
        oa, ra, da, ia = auto.step(acts[t])
        om, rm, dm, im = manual.step(acts[t])
        assert torch.equal(ra, rm) and torch.equal(da, dm) and torch.equal(ia["success"], im["success"]), t
        assert bool(da.all()) == ((t + 1) % horizon == 0), t
        if bool(dm.all()):
            om = manual.reset()
        assert torch.equal(oa, om), t
    sa, sm = state_arrays(auto), state_arrays(manual)
    for k in sa:
        assert np.array_equal(sa[k], sm[k]), k
    assert torch.equal(auto.num_interventions, manual.num_interventions)
    assert int(auto.num_interventions.min()) == int(auto.num_interventions.max()) == 1 + steps // horizon
    assert torch.equal(auto.steps_since_reset, manual.steps_since_reset)
    return auto, manual


@pytest.mark.parametrize("name", list(DOOR_PEG))
def test_auto_reset_matches_manual_reset_door_peg(name):
    auto, manual = compare_auto_and_manual(name, 256, 7, 3 * 7 + 2)
    if auto.env._eval_stats:
        assert torch.equal(auto.eval_stats(), manual.eval_stats())


@pytest.mark.parametrize("name", list(KITCHEN))
def test_auto_reset_matches_manual_reset_kitchen(name):
    compare_auto_and_manual(name, 48, 5, 3 * 5 + 1)


def test_kitchen_auto_reset_without_the_redo_path(monkeypatch):
    monkeypatch.setenv("EARL_MJ_REDO", "0")
    compare_auto_and_manual("kitchen-all_pairs", 24, 4, 9)


def test_lifelong_door_auto_reset_keeps_the_lifelong_return():
    def lifelong(auto):
        env = make("door-sparse", 6, 64, 5, auto_reset=auto)
        env.env._configure(lifelong=True, goal_change_frequency=4)
        return env
    auto, manual = lifelong(True), lifelong(False)
    assert torch.equal(auto.reset(), manual.reset())
    acts = actions("door-sparse", 64, 15, 9)
    for t in range(15):
        oa, ra, _, _ = auto.step(acts[t])
        om, rm, dm, _ = manual.step(acts[t])
        assert torch.equal(ra, rm)
        if bool(dm.all()):
            om = manual.reset()
        assert torch.equal(oa, om), t
    assert torch.equal(auto.env._counters(want_ll=True)[3], manual.env._counters(want_ll=True)[3])


@pytest.mark.parametrize("name", ["door-sparse", "peg-wide_init", "kitchen-all_pairs"])
def test_shards_reproduce_the_unsharded_auto_reset_env(name):
    n, horizon = 64 if name in KITCHEN else 200, 4 if name in KITCHEN else 6
    steps = 2 * horizon + 1
    full = make(name, horizon, n, 11, auto_reset=True)
    parts = [(0, n // 2), (n // 2, n - n // 2)]
    shards = [make(name, horizon, m, 11, auto_reset=True, env_offset=lo, total_envs=n) for lo, m in parts]
    of = full.reset()
    os_ = [s.reset() for s in shards]
    acts = actions(name, n, steps, 12)
    for t in range(steps + 1):
        for (lo, m), o in zip(parts, os_):
            assert torch.equal(of[lo:lo + m], o), t
        if t == steps:
            break
        of, rf, df, _ = full.step(acts[t])
        outs = [s.step(acts[t, lo:lo + m].contiguous()) for s, (lo, m) in zip(shards, parts)]
        for (lo, m), (o, r, d, _) in zip(parts, outs):
            assert torch.equal(rf[lo:lo + m], r) and torch.equal(df[lo:lo + m], d), t
        os_ = [o for o, _, _, _ in outs]
    for s, (lo, m) in zip(shards, parts):
        assert torch.equal(s.num_interventions, full.num_interventions[lo:lo + m])


@pytest.mark.parametrize("name", ["door-sparse", "peg-sparse", "kitchen-all_pairs"])
def test_host_path_matches_device_path_on_auto_reset_handles(name):
    n, horizon = (24, 3) if name in KITCHEN else (128, 5)
    steps = 2 * horizon + 2
    dev_env, host_env = make(name, horizon, n, 7, auto_reset=True), make(name, horizon, n, 7, auto_reset=True)
    dev_env.reset(), host_env.reset()
    acts = actions(name, n, steps, 8)
    for t in range(steps):
        od, rd, dd, _ = dev_env.step(acts[t])
        oh, rh, dh, _ = host_env.step(acts[t].cpu().numpy())
        assert isinstance(oh, np.ndarray)
        assert np.array_equal(od.cpu().numpy(), oh) and np.array_equal(rd.cpu().numpy(), rh), t
        assert np.array_equal(dd.cpu().numpy(), np.asarray(dh, bool)), t
    assert torch.equal(dev_env.num_interventions, host_env.num_interventions)


@pytest.mark.parametrize("name", ["door-sparse", "peg-sparse", "peg-reset_at_goal"])
def test_auto_reset_uses_the_goal_a_manual_reset_would_use(name):
    n, horizon = 64, 5
    auto, manual = make(name, horizon, n, 2, auto_reset=True), make(name, horizon, n, 2)
    auto.reset(), manual.reset()
    custom = (sawyer_door.initial_states if name.startswith("door") else sawyer_peg.initial_states)[0]
    auto.reset_goal(custom), manual.reset_goal(custom)
    acts = actions(name, n, horizon, 4)
    for t in range(horizon):
        oa, _, da, _ = auto.step(acts[t])
        manual.step(acts[t])
    assert bool(da.all())
    om = manual.reset()
    assert torch.equal(oa, om)
    assert np.array_equal(auto.goal, manual.goal)
    if name.startswith("door"):   # the door keeps the goal reset_goal() set
        assert torch.equal(oa[:, 7:14], torch.from_numpy(np.tile(custom, (n, 1))).to(oa))


def test_kitchen_redone_steps_at_the_horizon():
    """Contact-rich scripted policy of test_redo_scheduling_does_not_change_the_kitchen_physics: done steps whose envs the
    extra-large set re-stepped are reset after the redo kernel has written them."""
    n, horizon, steps = 592, 20, 3 * 20 + 1   # the arms reach the cabinet handle within the first horizon
    k = kitchen.REWARD_SITES.index("slide_site")
    auto, manual = make("kitchen-all_pairs", horizon, n, 4, auto_reset=True), make("kitchen-all_pairs", horizon, n, 4)
    auto.reset(), manual.reset()
    gen = torch.Generator(device=DEV)
    gen.manual_seed(8)
    redone_at_done = 0
    for t in range(steps):
        st = auto.get_state()
        d = torch.from_numpy(st["site_xpos"][:, k] - st["mocap_pos"]).to(DEV, torch.float32)
        u = torch.zeros((n, 9), device=DEV)
        u[:, :3] = torch.clamp(d * 10, -1, 1) * 0.5
        u += 0.1 * (torch.rand((n, 9), generator=gen, device=DEV) * 2 - 1)
        before = auto.work_counters()["redone_states"]
        oa, ra, da, _ = auto.step(u)
        om, rm, dm, _ = manual.step(u)
        if bool(da.all()):
            redone_at_done += auto.work_counters()["redone_states"] - before
        if bool(dm.all()):
            om = manual.reset()
        assert torch.equal(ra, rm) and torch.equal(da, dm) and torch.equal(oa, om), t
    wa, wm = auto.work_counters(), manual.work_counters()
    if redone_at_done == 0:
        pytest.skip("the scripted reach no longer outgrows the primary capacity set at the horizon")
    assert wa["overflow_states"] == 0 and wm["overflow_states"] == 0
    assert wa["redone_states"] == wm["redone_states"]
    sa, sm = auto.get_state(), manual.get_state()
    for key in sa:
        assert np.array_equal(sa[key], sm[key]), key


@pytest.mark.parametrize("name", ["sawyer_door", "sawyer_peg", "kitchen"])
def test_loader_resets_the_train_env_at_the_horizon(name):
    horizon = 4
    reward = "dense" if name == "kitchen" else "sparse"
    tr, ev = eb.EARLEnvs(name, reward_type=reward, auto_reset=True, train_horizon=horizon, eval_horizon=horizon,
                         num_envs=8, device=DEV).get_envs()
    tr.reset(), ev.reset()
    a = torch.zeros((8, 9 if name == "kitchen" else 4), device=DEV)
    for t in range(1, horizon + 2):
        _, _, dt, _ = tr.step(a)
        _, _, de, _ = ev.step(a)
        assert bool(dt.all()) == (t == horizon)
        assert bool(de.all()) == (t >= horizon)            # the eval env does not reset
    assert tr.num_interventions.tolist() == [2] * 8 and tr.steps_since_reset.tolist() == [1] * 8
    assert ev.num_interventions.tolist() == [1] * 8 and ev.steps_since_reset.tolist() == [horizon + 1] * 8


@pytest.mark.parametrize("name", ["door-sparse", "peg-dense"])
def test_launches_per_step(name):
    """step kernel + concurrent redo kernel + order kernel; auto reset adds exactly the reset pass"""
    for auto, want in ((False, 3), (True, 4)):
        env = make(name, 1000, 64, auto_reset=auto)
        env.reset()
        a = actions(name, 64, 5, 1)
        l0 = env.launch_count
        for t in range(5):
            env.step(a[t])
        assert env.launch_count - l0 == 5 * want, auto
