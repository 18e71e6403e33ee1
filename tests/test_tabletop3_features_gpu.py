"""Three-object tabletop auto-reset, evaluation statistics and sharding on the B200: the reset fused into the step equals a
masked reset() after done, bit for bit; the whole feature set against the test oracle; the chunked host path; shards
against the unsharded env.  Dense rewards within 2e-6 relative of the oracle (as in test_tabletop3_gpu.py), dense
returns within 1e-9 relative; everything else exact."""
import ctypes

import numpy as np
import pytest
import torch

from earl_benchmark_b200 import _lib, shard_range
from earl_benchmark_b200.envs import tabletop_manipulation_3obj as tt3
from earl_benchmark_b200.wrappers.persistent_state_wrapper import PersistentStateWrapper
from tabletop3_features_oracle import Tabletop3FeaturesOracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEED = 7


def make(n, horizon, seed=SEED, **kw):
    return PersistentStateWrapper(tt3.TabletopManipulation(num_envs=n, device=DEV, seed=seed, **kw), horizon)


def actions(rs, steps, n):
    a = rs.uniform(-1.2, 1.2, (steps, n, 3)).astype(np.float32)
    a[:, : n // 2, 2] = np.where(rs.uniform(size=(steps, n // 2)) < 0.9, 1.0, -1.0)
    return a


def np_(x):
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


CASES = {
    "sparse": dict(reward_type="sparse"),
    "dense": dict(reward_type="dense"),
    "eval_stats": dict(reward_type="sparse", eval_stats=True),
    "reset_at_goal": dict(reward_type="sparse", reset_at_goal=True, reset_stream_rows=3),
}


@pytest.mark.parametrize("case", list(CASES))
def test_auto_reset_equals_manual_masked_reset(case):
    n, horizon = 5003, 9
    steps = 8 * horizon + 4                    # > 7 horizons: with R = 3 every cursor wraps
    kw = CASES[case]
    auto, man = make(n, horizon, auto_reset=True, **kw), make(n, horizon, **kw)
    rows = tt3.reset_stream(SEED, n, 0, n, 3) if kw.get("reset_at_goal") else None
    cursor = np.zeros(n, np.int64)

    def man_reset(mask):
        """the manual handle takes the same stream rows as init_qpos, through a host cursor"""
        if rows is None:
            return man.reset(mask=mask)
        sel = np_(mask).astype(bool)
        q = rows[cursor % len(rows), np.arange(n)]
        cursor[sel] += 1
        return man.reset(mask=mask, init_qpos=q)

    assert torch.equal(auto.reset(), man.reset())   # stream row 0 is the first full host reset
    cursor[:] = 1
    rs = np.random.RandomState(5)
    acts = torch.from_numpy(actions(rs, steps, n)).to(DEV)
    half = torch.from_numpy(np.arange(n) % 2 == 0).to(DEV)
    resets = 0
    for t in range(steps):
        if t == horizon // 2:                    # stagger the episodes
            assert torch.equal(auto.reset(mask=half), man_reset(half))
        before = auto.launch_count
        oa, ra, da, ia = auto.step(acts[t])
        assert auto.launch_count == before + 1   # the reset is fused: one kernel per step
        om, rm, dm, im = man.step(acts[t])
        assert torch.equal(ra, rm) and torch.equal(da, dm) and torch.equal(ia["success"], im["success"]), t
        if bool(dm.any()):
            resets += 1
            om = man_reset(dm)
        assert torch.equal(oa, om), t
    assert resets >= 8
    qa, aa = auto.get_state()
    qm, am = man.get_state()
    assert torch.equal(qa, qm) and torch.equal(aa, am)
    assert auto.total_steps == man.total_steps == steps
    assert torch.equal(auto.num_interventions, man.num_interventions)
    assert torch.equal(auto.steps_since_reset, man.steps_since_reset)
    if kw.get("eval_stats"):
        assert torch.equal(auto.eval_stats(), man.eval_stats())
    if rows is not None:
        assert cursor.min() > 3


def check_stats(env, orc, dense):
    got, want = np_(env.eval_stats()), orc.eval_stats()
    assert np.array_equal(got[1:], want[1:])
    if dense:
        assert abs(got[0] - want[0]) <= 1e-9 * abs(want[0])
    else:
        assert got[0] == want[0]


@pytest.mark.parametrize("case", ["sparse", "dense", "reset_at_goal"])
def test_auto_reset_and_eval_stats_against_the_oracle(case):
    n, horizon, steps = 5003, 20, 110
    dense = case == "dense"
    rag = case == "reset_at_goal"
    rs = np.random.RandomState(13)
    env = make(n, horizon, reward_type="dense" if dense else "sparse", reset_at_goal=rag, reset_stream_rows=4,
               auto_reset=True, eval_stats=True)
    rows = tt3.reset_stream(SEED, n, 0, n, 4) if rag else None
    orc = Tabletop3FeaturesOracle(n, horizon, dense=dense, auto_reset=True, reset_rows=rows)
    if rag:
        assert np.array_equal(np_(env.reset()), orc.reset())
    else:   # objects scattered around the fist so all three get grasped and dragged
        q0 = np.concatenate([rs.uniform(-2, 2, (n, 2))] * 4, axis=1) + np.concatenate([np.zeros((n, 2)), rs.uniform(-0.6, 0.6, (n, 6))], axis=1)
        assert np.array_equal(np_(env.reset(init_qpos=q0)), orc.reset(init_qpos=q0))
    acts = actions(rs, steps, n)
    stagger = np.arange(n) % 3 == 0
    successes = 0
    for t in range(steps):
        if t == 7:
            assert np.array_equal(np_(env.reset(mask=stagger)), orc.reset(mask=stagger))
            check_stats(env, orc, dense)         # a masked reset clears the statistics of its envs
        if t % 3 == 2:
            o, r, d, info = env.step(acts[t])   # host path (numpy in, numpy out)
            s = info["success"]
        else:
            o, r, d, info = env.step(torch.from_numpy(acts[t]).to(DEV))
            o, r, d, s = np_(o), np_(r), np_(d), np_(info["success"])
        o2, r2, d2, s2 = orc.step(acts[t])
        assert np.array_equal(o, o2) and np.array_equal(d, d2) and np.array_equal(s, s2), t
        if dense:
            assert np.allclose(r, r2, rtol=2e-6, atol=2e-6), t
        else:
            assert np.array_equal(r.astype(np.float64), r2), t
        successes += int(s2.sum())
        if t % 10 == 9:
            check_stats(env, orc, dense)
    q, att = env.get_state()
    assert np.array_equal(np_(q), orc.qpos) and np.array_equal(np_(att), orc.att)
    assert np.array_equal(np_(env.num_interventions), orc.num_interventions)
    assert np.array_equal(np_(env.steps_since_reset), orc.steps_since_reset)
    assert orc.num_interventions.min() >= 1 + (steps - 7) // horizon
    if rag:   # resets near the goal: the success counts are exercised (from the scattered start nothing succeeds)
        assert successes > 0
    env.reset()
    orc.reset()
    check_stats(env, orc, dense)
    assert np_(env.eval_stats()).tolist() == [0.0, 0.0, 0.0, float(n)]


def test_chunked_host_path_with_auto_reset_from_the_stream():
    n, horizon, steps = 2 * 2**18 + 2051, 5, 13   # two host chunks; R = 2 wraps after the second auto-reset
    kw = dict(reward_type="sparse", reset_at_goal=True, reset_stream_rows=2, auto_reset=True, eval_stats=True)
    host, dev = make(n, horizon, **kw), make(n, horizon, **kw)
    assert np.array_equal(np_(host.reset()), np_(dev.reset()))
    rs = np.random.RandomState(2)
    for t in range(steps):
        a = actions(rs, 1, n)[0]
        before = host.launch_count
        oh, rh, dh, ih = host.step(a)
        assert host.launch_count - before == 2      # one launch per chunk
        od, rd, dd, idd = dev.step(torch.from_numpy(a).to(DEV))
        assert np.array_equal(oh, np_(od)) and np.array_equal(rh, np_(rd)), t
        assert np.array_equal(dh, np_(dd)) and np.array_equal(ih["success"], np_(idd["success"])), t
        assert bool(dh.all()) == ((t + 1) % horizon == 0), t
    assert torch.equal(host.get_state()[0], dev.get_state()[0])
    assert torch.equal(host.eval_stats(), dev.eval_stats())


@pytest.mark.parametrize("auto_reset", [False, True])
def test_shards_reproduce_the_unsharded_env(auto_reset):
    total, horizon = 1001, 6
    kw = dict(reward_type="sparse", reset_at_goal=True, eval_stats=True, auto_reset=auto_reset)
    spans = [shard_range(total, r, 3) for r in range(3)]
    whole = make(total, horizon, **kw)
    shards = [make(hi - lo, horizon, env_offset=lo, total_envs=total, **kw) for lo, hi in spans]
    for _ in range(2):   # successive full resets draw the same rows of the job's stream
        ow = whole.reset()
        assert torch.equal(torch.cat([s.reset() for s in shards]), ow)
    rs = np.random.RandomState(3)
    steps = 3 * horizon + 2 if auto_reset else horizon
    acts = torch.from_numpy(actions(rs, steps, total)).to(DEV)
    for t in range(steps):
        ow, rw, dw, iw = whole.step(acts[t])
        outs = [s.step(acts[t, lo:hi].contiguous()) for s, (lo, hi) in zip(shards, spans)]
        for k, ref in enumerate((ow, rw, dw, iw["success"])):
            part = [o[k] if k < 3 else o[3]["success"] for o in outs]
            assert torch.equal(torch.cat(part), ref), (t, k)
    assert torch.equal(sum(s.eval_stats() for s in shards), whole.eval_stats())


def test_plain_handles_keep_the_plain_step_kernel():
    from torch.profiler import ProfilerActivity, profile
    a = torch.zeros((300, 3), device=DEV)
    for kw, general in (({}, "false"), ({"reward_type": "dense"}, "false"), ({"eval_stats": True}, "true"),
                        ({"auto_reset": True}, "true")):
        env = make(300, 50, **kw)
        env.reset()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            env.step(a)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if "tt3_step_kernel" in e.name]
        assert names and all(f"tt3_step_kernel<{general}>" in k for k in names), (kw, names)


def test_stream_handle_rejects_work_before_its_stream():
    env = tt3.TabletopManipulation(num_envs=8, device=DEV, reset_at_goal=True, auto_reset=True)
    env._ensure()
    h = env._handle
    # a fresh handle with the same flags but no stream: reset without init_qpos and step are refused
    cfg = _lib.Tt3Config()
    cfg.num_envs, cfg.device, cfg.num_goals, cfg.episode_horizon = 8, 0, 1, 4
    cfg.flags = _lib.FLAG_AUTO_RESET | _lib.FLAG_RESET_AT_GOAL
    raw = ctypes.c_void_p()
    L = _lib.lib()
    _lib.check(L.earl_tt3_create(ctypes.byref(cfg), ctypes.sizeof(cfg), ctypes.byref(raw)))
    try:
        assert L.earl_tt3_reset(raw, None, None, None, None, None) == -1
        assert L.earl_tt3_set_reset_stream(h, np.zeros((5, 8, 8)).ctypes.data, 5) == -1   # R is fixed per handle
    finally:
        L.earl_tt3_destroy(raw)
    plain = tt3.TabletopManipulation(num_envs=8, device=DEV, auto_reset=True)
    plain._ensure()
    assert L.earl_tt3_set_reset_stream(plain._handle, np.zeros((2, 8, 8)).ctypes.data, 2) == -1
