"""final_obs=True on the B200, all five tasks.  Three handles step on the same seeds and actions: `auto` (auto-reset with the
flag), `plain` (auto-reset without it) and `manual` (no auto-reset, reset(mask=done) after each step).  On every step the
rows of the final-observation buffer where done is set equal, bit for bit, the observation `manual` returned before its
reset; every other row keeps what it held (NaN until an env's first episode ends); every output, state, counter and
statistic of `auto` equals that of `plain`; and the flag costs the door / peg one launch per step and the tabletops none."""
import numpy as np
import pytest
import torch

from earl_benchmark_b200 import _lib, shard_range
from earl_benchmark_b200.envs import kitchen, sawyer_door, sawyer_peg, tabletop_manipulation as tt
from earl_benchmark_b200.envs import tabletop_manipulation_3obj as tt3
from earl_benchmark_b200.wrappers.persistent_state_wrapper import PersistentStateWrapper

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
R = 64   # rows of the pre-drawn reset streams (the constructors' default)

CASES = {
    "tt-f32-sparse": ("tt", dict(reward_type="sparse")),
    "tt-f32-dense": ("tt", dict(reward_type="dense")),
    "tt-f64-sparse": ("tt", dict(reward_type="sparse", state_dtype="float64")),
    "tt-f64-dense": ("tt", dict(reward_type="dense", state_dtype="float64", eval_stats=True)),
    "tt-lifelong": ("tt", dict(reward_type="sparse", lifelong=3, eval_stats=True)),
    "tt-per_env_goals": ("tt", dict(reward_type="dense", per_env_goals=True)),
    "tt-f64-per_env_goals-lifelong": ("tt", dict(reward_type="sparse", state_dtype="float64", per_env_goals=True, lifelong=4)),
    "tt-reset_at_goal": ("tt", dict(reward_type="sparse", reset_at_goal=True)),
    "tt3-sparse": ("tt3", dict(reward_type="sparse")),
    "tt3-dense": ("tt3", dict(reward_type="dense")),
    "tt3-reset_at_goal": ("tt3", dict(reward_type="sparse", reset_at_goal=True, reset_stream_rows=3)),
    "tt3-eval_stats": ("tt3", dict(reward_type="dense", eval_stats=True)),
    "door-sparse": ("door", dict(reward_type="sparse", eval_stats=True)),
    "door-dense": ("door", dict(reward_type="dense")),
    "door-reset_at_goal": ("door", dict(reset_at_goal=True)),
    "door-lifelong": ("door", dict(lifelong=4)),
    "peg-sparse": ("peg", dict(reward_type="sparse", eval_stats=True)),
    "peg-dense": ("peg", dict(reward_type="dense")),
    "peg-reset_at_goal": ("peg", dict(reset_at_goal=True)),
    "peg-wide_init": ("peg", dict(wide_init=True)),
    "kitchen-all_pairs": ("kitchen", dict(task="all_pairs", eval_stats=True)),
    "kitchen-microwave": ("kitchen", dict(task="microwave")),
}
ACT = {"tt": 3, "tt3": 3, "door": 4, "peg": 4, "kitchen": 9}
EXTRA_LAUNCHES = {"tt": 0, "tt3": 0, "door": 1, "peg": 1}   # per step, flagged against plain (kitchen counts no launches)


def make(kind, n, horizon, seed, auto_reset, final_obs=False, lifelong=None, **kw):
    kw = dict(kw, num_envs=n, device=DEV, seed=seed, auto_reset=auto_reset)
    if final_obs:
        kw["final_obs"] = True
    cls = {"tt": tt.TabletopManipulation, "tt3": tt3.TabletopManipulation, "door": sawyer_door.SawyerDoorV2,
           "peg": sawyer_peg.SawyerPegV2, "kitchen": kitchen.Kitchen}[kind]
    env = PersistentStateWrapper(cls(**kw), horizon)
    if lifelong:
        env.env._configure(lifelong=True, goal_change_frequency=lifelong)
    return env


class Manual:
    """reset(mask) of the handle without auto-reset, fed the draws the auto-reset handles take from their pre-drawn stream"""

    def __init__(self, env, kind, opts, n, seed, total=None, offset=0):
        self.env, self.kind, self.n = env, kind, n
        total = n if total is None else total
        self.cursor = np.ones(n, np.int64)   # the first full reset takes row 0 on every handle
        self.rows = None
        if kind == "tt3" and opts.get("reset_at_goal"):
            self.rows = tt3.reset_stream(seed, total, offset, n, opts["reset_stream_rows"])
        elif kind == "door":
            self.rows = sawyer_door.reset_stream(seed, total, offset, n, R, opts.get("reset_at_goal", False))[..., 0]
        elif kind == "peg":
            self.goal_rows, self.rows = sawyer_peg.reset_stream(seed, total, offset, n, R, opts.get("reset_at_goal", False),
                                                                opts.get("wide_init", False))
        elif kind == "kitchen" and opts["task"] == "all_pairs":
            self.rows = kitchen.reset_stream(seed, total, offset, n, R, "all_pairs")[0]

    def reset(self, mask):
        sel = mask.cpu().numpy().astype(bool)
        if self.rows is None:
            return self.env.reset(mask=mask)
        e = self.cursor % len(self.rows)
        self.cursor[sel] += 1
        if self.kind == "kitchen":
            return self.env.reset(mask=mask, config_index=self.rows[e, np.arange(self.n)][sel])
        draw = self.rows[e, np.arange(self.n)]
        if self.kind == "tt3":
            return self.env.reset(mask=mask, init_qpos=draw)
        if self.kind == "door":
            return self.env.reset(mask=mask, door_angle=draw)
        g = self.env.env._goal_rows
        g[mask.bool()] = torch.from_numpy(self.goal_rows[e, np.arange(self.n)]).to(g)[mask.bool()]
        return self.env.reset(mask=mask, peg_pos=draw)


def bits(t):
    return t.view(torch.int64 if t.dtype == torch.float64 else torch.int32)


def snapshot(env):
    """every output of a handle besides the step's own: state, counters, statistics, lifelong return, goals"""
    base = env.env
    st = base.get_state()
    out = {k: np.asarray(v) for k, v in st.items()} if isinstance(st, dict) else {f"s{k}": v.cpu().numpy() for k, v in enumerate(st)}
    total, interv, since, ll = base._counters(want_ll=getattr(base, "_lifelong", False))
    out.update(total=np.array(total), interv=interv.cpu().numpy(), since=since.cpu().numpy())
    if ll is not None:
        out["ll"] = ll.cpu().numpy()
    if getattr(base, "_eval_stats", False):
        out["eval"] = base.eval_stats().cpu().numpy()
    if getattr(base, "_per_env_goals", False):
        out["goals"] = base.get_goals().cpu().numpy()
    if hasattr(base, "_goal_rows") and isinstance(base._goal_rows, torch.Tensor):
        out["goal_rows"] = base._goal_rows.cpu().numpy()
    return out


def run_three(name, n, horizon, steps, seed=5, stagger=True):
    kind, opts = CASES[name]
    auto = make(kind, n, horizon, seed, True, final_obs=True, **opts)
    plain = make(kind, n, horizon, seed, True, **opts)
    man_env = make(kind, n, horizon, seed, False, **opts)
    man = Manual(man_env, kind, opts, n, seed)
    oa, op, om = auto.reset(), plain.reset(), man_env.reset()
    assert torch.equal(oa, op) and torch.equal(oa, om)
    fin = auto.env._final_obs
    expect = torch.full_like(fin, float("nan"))
    assert torch.equal(bits(fin), bits(expect))
    gen = torch.Generator(device=DEV)
    gen.manual_seed(seed)
    acts = torch.rand((steps, n, ACT[kind]), generator=gen, device=DEV) * 2.4 - 1.2
    idx = torch.arange(n, device=DEV)
    keep = idx % 4 == 0          # reset every horizon - 1 steps: these envs never end an episode
    late = idx % 4 == 1          # one masked reset early on: their episodes end off the common beat
    ever = torch.zeros(n, dtype=torch.bool, device=DEV)
    extra = EXTRA_LAUNCHES.get(kind)
    la0, lp0 = (auto.launch_count, plain.launch_count) if extra is not None else (0, 0)
    for t in range(steps):
        for mask, when in ((keep, t % (horizon - 1) == horizon - 2), (late, t == horizon // 2)):
            if stagger and when:
                oa, op, om = auto.reset(mask=mask), plain.reset(mask=mask), man.reset(mask)
                assert torch.equal(oa, op) and torch.equal(oa, om), t
        if opts.get("per_env_goals") and t == 1:
            goals = torch.rand((n, 6 if kind == "tt" else 7), generator=gen, device=DEV) * 4 - 2
            for env in (auto, plain, man_env):
                env.set_goals(goals, mask=idx % 3 == 0)
        oa, ra, da, ia = auto.step(acts[t])
        op, rp, dp, ip = plain.step(acts[t])
        om, rm, dm, im = man_env.step(acts[t])
        assert "final_observation" not in ip and ia["final_observation"] is fin
        assert torch.equal(oa, op) and torch.equal(ra, rp) and torch.equal(da, dp), t
        assert torch.equal(ia["success"], ip["success"]), t
        assert torch.equal(ra, rm) and torch.equal(da, dm) and torch.equal(ia["success"], im["success"]), t
        expect[da] = om[da]
        ever |= da
        assert torch.equal(bits(fin), bits(expect)), t
        if bool(dm.any()):   # what a training loop keeps: the reset rows of reset(), the step's rows elsewhere (a Sawyer
            # reset recomputes the other rows from a fresh kinematics pass, which need not match the step's bits)
            om = torch.where(dm.view(-1, 1), man.reset(dm), om)
        assert torch.equal(oa, om), t
    assert bool(ever.any()) and not bool(ever[keep].any() if stagger else False)
    assert bool(torch.isnan(fin[~ever]).all()) and not bool(torch.isnan(fin[ever]).any())
    sa, sp = snapshot(auto), snapshot(plain)
    assert sa.keys() == sp.keys()
    for k in sa:
        assert np.array_equal(sa[k], sp[k]), k
    if extra is not None:
        assert (auto.launch_count - la0) - (plain.launch_count - lp0) == extra * steps
    return auto, plain


SIZES = {"tt": (1000, 7, 40), "tt3": (1003, 6, 34), "door": (96, 5, 21), "peg": (96, 5, 21), "kitchen": (24, 4, 13)}


@pytest.mark.parametrize("name", list(CASES))
def test_final_observation_equals_the_observation_before_the_reset(name):
    run_three(name, *SIZES[CASES[name][0]])


@pytest.mark.parametrize("name", ["kitchen-all_pairs", "kitchen-microwave"])
def test_kitchen_without_the_redo_path(name, monkeypatch):
    monkeypatch.setenv("EARL_MJ_REDO", "0")
    run_three(name, 24, 4, 9)


def test_tabletop_at_scale():
    run_three("tt-f32-sparse", 1 << 20, 64, 200, stagger=False)


@pytest.mark.parametrize("name", ["door-sparse", "peg-sparse"])
def test_door_peg_at_scale(name):
    run_three(name, 4096, 6, 13, stagger=False)


@pytest.mark.parametrize("name", ["tt-f32-dense", "tt-f64-sparse", "tt3-reset_at_goal", "door-sparse", "kitchen-all_pairs"])
def test_host_step_matches_the_device_step(name):
    kind, opts = CASES[name]
    n, horizon = (24, 3) if kind == "kitchen" else ((64, 4) if kind in ("door", "peg") else (2 * 2**18 + 2051, 5))
    steps = 2 * horizon
    dev_env = make(kind, n, horizon, 7, True, final_obs=True, **opts)
    host_env = make(kind, n, horizon, 7, True, final_obs=True, **opts)
    dev_env.reset(), host_env.reset()
    gen = torch.Generator(device=DEV)
    gen.manual_seed(3)
    for t in range(steps):
        a = torch.rand((n, ACT[kind]), generator=gen, device=DEV) * 2 - 1
        od, rd, dd, idd = dev_env.step(a)
        oh, rh, dh, ih = host_env.step(a.cpu().numpy())
        assert isinstance(ih["final_observation"], np.ndarray)
        assert np.array_equal(od.cpu().numpy(), oh) and np.array_equal(dd.cpu().numpy(), np.asarray(dh, bool)), t
        fd, fh = idd["final_observation"].cpu().numpy(), ih["final_observation"]
        assert np.array_equal(fd.view(np.uint8), fh.view(np.uint8)), t
    assert bool(dd.all())


@pytest.mark.parametrize("name", ["tt-f32-sparse", "tt3-reset_at_goal", "door-sparse", "peg-wide_init", "kitchen-all_pairs"])
def test_two_shards_equal_one_handle(name):
    kind, opts = CASES[name]
    total, horizon = (48, 4) if kind == "kitchen" else ((128, 5) if kind in ("door", "peg") else (1001, 6))
    steps = 2 * horizon
    whole = make(kind, total, horizon, 11, True, final_obs=True, **opts)
    spans = [shard_range(total, r, 2) for r in range(2)]
    shards = [make(kind, hi - lo, horizon, 11, True, final_obs=True, env_offset=lo, total_envs=total, **opts) for lo, hi in spans]
    ow = whole.reset()
    assert torch.equal(torch.cat([s.reset() for s in shards]), ow)
    gen = torch.Generator(device=DEV)
    gen.manual_seed(4)
    for t in range(steps):
        a = torch.rand((total, ACT[kind]), generator=gen, device=DEV) * 2 - 1
        ow, _, dw, iw = whole.step(a)
        outs = [s.step(a[lo:hi].contiguous()) for s, (lo, hi) in zip(shards, spans)]
        assert torch.equal(torch.cat([o[0] for o in outs]), ow) and torch.equal(torch.cat([o[2] for o in outs]), dw), t
        assert torch.equal(bits(torch.cat([o[3]["final_observation"] for o in outs])), bits(iw["final_observation"])), t
    assert bool(dw.all())


@pytest.mark.parametrize("kind,opts", [("tt", dict(reward_type="sparse")), ("tt3", dict(reward_type="sparse")),
                                       ("door", dict()), ("kitchen", dict(task="microwave"))])
def test_errors(kind, opts, monkeypatch):
    L = _lib.lib()
    n = 16
    a = torch.zeros((n, ACT[kind]), device=DEV)
    # the flag without auto-reset: refused by the constructor, and by the library for a config that asks for it anyway
    with pytest.raises(ValueError):
        make(kind, n, 4, 1, False, final_obs=True, **opts)
    # registering a buffer on a handle without the flag
    plain = make(kind, n, 4, 1, True, **opts)
    plain.reset()
    setter = {"tt": "earl_set_final_obs", "tt3": "earl_tt3_set_final_obs", "door": "earl_mj_set_final_obs",
              "kitchen": "earl_mjk_set_final_obs"}[kind]
    buf = torch.zeros((n, 46 if kind == "kitchen" else 20), dtype=torch.float64 if kind == "kitchen" else torch.float32, device=DEV)
    assert getattr(L, setter)(plain.env._handle, buf.data_ptr()) == -1
    assert b"EARL_FLAG_FINAL_OBS" in L.earl_last_error()
    # stepping a flagged handle before a buffer is registered (the env's own registration skipped)
    monkeypatch.setattr(L, setter, lambda h, p: 0)
    bare = make(kind, n, 4, 1, True, final_obs=True, **opts)
    bare.reset()
    with pytest.raises(_lib.EarlError) as ei:
        bare.step(a)
    assert ei.value.code == -1 and "before the first step" in str(ei.value)
    if kind in ("tt", "tt3"):
        with pytest.raises(_lib.EarlError):
            bare.step(a.cpu().numpy())
    monkeypatch.undo()
    # rollouts of a flagged handle: refused by the env and by the library
    if kind in ("tt", "tt3"):
        env = make(kind, n, 4, 1, True, final_obs=True, **opts)
        env.reset()
        od = tt.OBS_DIM if kind == "tt" else tt3.OBS_DIM
        acts = torch.zeros((2, n, 3), device=DEV)
        obs, rew, done = torch.empty((2, n, od), device=DEV), torch.empty((2, n), device=DEV), torch.empty((2, n), dtype=torch.uint8, device=DEV)
        with pytest.raises(RuntimeError):
            env.rollout_into(acts, 2, obs, rew, done)
        fn = L.earl_rollout if kind == "tt" else L.earl_tt3_rollout
        assert fn(env.env._handle, acts.data_ptr(), 2, 2, obs.data_ptr(), rew.data_ptr(), done.data_ptr(), None, 2, None) == -1
        assert env.total_steps == 0
