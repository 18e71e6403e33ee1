#!/usr/bin/env python
"""What per-env goals (`per_env_goals=True`, set_goals / get_goals) cost, random actions, one GPU.

tabletop_manipulation at --tabletop-envs (default 1M and 4M), modes alternated window by window in one process:
  fast            default sparse handle (the FAST step kernel)
  general         default dense handle (the general step kernel)
  goals-{sparse,dense}-none   per_env_goals handle (the GOALS step kernel), goals never changed
  goals-{sparse,dense}-400    the same with set_goals() of every env every 400 steps
  goals-{sparse,dense}-1      the same with set_goals() of every env every step
sawyer_door / sawyer_peg at --sawyer-envs (default 65,536): default, goals-none, goals-1 and goals-600, one window of
--sawyer-steps (600) steps each, after the same warm-up, in the same process.
Also: one set_goals() call (CUDA events around --calls back-to-back calls), and the copy rate of a 2 GiB
device-to-device torch copy as the HBM reference, against which the tabletop GOALS kernel's algorithmic bytes
(146 B per env step: the general kernel's 114 B plus the 32-byte goal slot it reads) are set.
Windows of the tabletop modes last at least --min-window seconds, timed with CUDA events.  Prints one JSON line per
measurement and writes them, with the GPU's name and power limit, to --out.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from earl_benchmark_b200.envs import sawyer_door, sawyer_peg  # noqa: E402
from earl_benchmark_b200.envs.tabletop_manipulation import TabletopManipulation  # noqa: E402
from earl_benchmark_b200.wrappers.persistent_state_wrapper import PersistentStateWrapper  # noqa: E402

DEV = "cuda:0"
NEVER = 1 << 40
TT_BYTES = {"fast": 114, "general": 114, "goals": 146}   # algorithmic HBM bytes per env step with a success output
TT_MODES = ("fast", "general", "goals-sparse-none", "goals-sparse-400", "goals-sparse-1",
            "goals-dense-none", "goals-dense-400", "goals-dense-1")
SAWYER_MODES = ("default", "goals-none", "goals-600", "goals-1")


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
    except (OSError, subprocess.CalledProcessError):
        name, power = torch.cuda.get_device_name(0), "unknown"
    return {"gpu": name, "power_limit": power}


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def copy_peak():
    """bytes moved (read + write) per second by a 2 GiB device-to-device copy, best of 10"""
    src = torch.empty(1 << 31, dtype=torch.uint8, device=DEV)
    dst = torch.empty_like(src)
    dst.copy_(src)
    ms = min(timed(lambda: dst.copy_(src)) for _ in range(10))
    return 2 * src.numel() / (ms * 1e-3)


def goal_batches(n, width, count, seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return [torch.rand((n, width), generator=g, device=DEV) * 4 - 2 for _ in range(count)]


def run(env, acts, goals, every, t0, steps):
    ring = len(acts)
    for t in range(t0, t0 + steps):
        if every and t % every == 0:
            env.set_goals(goals[(t // every) % len(goals)])
        env.step(acts[t % ring])


def tt_env(mode, n):
    if mode == "fast":
        return TabletopManipulation(reward_type="sparse", num_envs=n, device=DEV, seed=1), 0
    if mode == "general":
        return TabletopManipulation(reward_type="dense", num_envs=n, device=DEV, seed=1), 0
    _, reward, every = mode.split("-")
    env = TabletopManipulation(reward_type=reward, num_envs=n, device=DEV, seed=1, per_env_goals=True)
    return env, {"none": 0, "400": 400, "1": 1}[every]


def bench_tabletop(n, rounds, min_window, calls, peak):
    acts = [torch.rand((n, 3), device=DEV) * 2 - 1 for _ in range(8)]     # 8 x 12 B x N: larger than L2 from 1M envs on
    goals = goal_batches(n, 6, 2, 7)
    envs = {}
    for m in TT_MODES:
        env, every = tt_env(m, n)
        env.reset()
        envs[m] = (env, every)
    clock = {m: 0 for m in TT_MODES}
    for m in TT_MODES:   # warm-up, and the window length from the slowest mode
        run(envs[m][0], acts, goals, envs[m][1], 0, 400)
        clock[m] = 400
    probe = min(timed(lambda m=m: run(envs[m][0], acts, goals, envs[m][1], clock[m], 400)) for m in TT_MODES)
    for m in TT_MODES:
        clock[m] += 400
    steps = 400 * max(1, int(-(-min_window * 1e3 // probe)))
    ms = {m: [] for m in TT_MODES}
    for _ in range(rounds):
        for m in TT_MODES:
            ms[m].append(timed(lambda m=m: run(envs[m][0], acts, goals, envs[m][1], clock[m], steps)))
            clock[m] += steps
    out = []
    for m in TT_MODES:
        rates = [n * steps / (t * 1e-3) for t in ms[m]]
        kind = m if m in TT_BYTES else "goals"
        byte_rate = max(rates) * TT_BYTES[kind]
        out.append(dict(task="tabletop_manipulation", mode=m, num_envs=n, steps_per_window=steps, windows=rounds,
                        env_steps_per_s=max(rates), env_steps_per_s_all=rates, bytes_per_env_step=TT_BYTES[kind],
                        algorithmic_bytes_per_s=byte_rate, fraction_of_copy_peak=byte_rate / peak))
    env = envs["goals-sparse-1"][0]
    env.set_goals(goals[0])
    t = min(timed(lambda: [env.set_goals(goals[k % 2]) for k in range(calls)]) for _ in range(3))
    out.append(dict(task="tabletop_manipulation", mode="set_goals_call", num_envs=n, calls=calls, us_per_call=t * 1e3 / calls))
    for env, _ in envs.values():
        env.close()
    return out


def bench_sawyer(task, n, steps, calls):
    cls = sawyer_door.SawyerDoorV2 if task == "sawyer_door" else sawyer_peg.SawyerPegV2
    g = torch.Generator(device=DEV)
    g.manual_seed(1234)
    acts = [torch.rand((n, 4), generator=g, device=DEV) * 2 - 1 for _ in range(64)]
    goals = [x * 0.1 + torch.tensor([0.0, 0.6, 0.2, 1.0, 0.0, 0.7, 0.1], device=DEV) for x in goal_batches(n, 7, 2, 9)]
    envs, every = {}, {"default": 0, "goals-none": 0, "goals-600": 600, "goals-1": 1}
    for m in SAWYER_MODES:
        env = PersistentStateWrapper(cls(reward_type="sparse", num_envs=n, device=DEV, seed=1, per_env_goals=m != "default"), NEVER)
        env.reset()
        run(env, acts, goals, every[m], 0, 20)
        envs[m] = env
    torch.cuda.synchronize()
    out = []
    for m in SAWYER_MODES:   # the same action sequence from the same reset for every mode
        t = timed(lambda m=m: run(envs[m], acts, goals, every[m], 20, steps))
        out.append(dict(task=task, mode=m, num_envs=n, steps_per_window=steps, windows=1, env_steps_per_s=n * steps / (t * 1e-3),
                        set_goals_calls=0 if not every[m] else -(-steps // every[m])))
    env = envs["goals-1"]
    t = min(timed(lambda: [env.set_goals(goals[k % 2]) for k in range(calls)]) for _ in range(3))
    out.append(dict(task=task, mode="set_goals_call", num_envs=n, calls=calls, us_per_call=t * 1e3 / calls))
    for env in envs.values():
        env.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tabletop-envs", type=int, nargs="*", default=[1 << 20, 1 << 22])
    ap.add_argument("--sawyer-tasks", nargs="*", default=["sawyer_door", "sawyer_peg"])
    ap.add_argument("--sawyer-envs", type=int, default=65536)
    ap.add_argument("--sawyer-steps", type=int, default=600)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--min-window", type=float, default=0.3, help="seconds")
    ap.add_argument("--calls", type=int, default=200, help="back-to-back set_goals() calls per timing")
    ap.add_argument("--out", default=None, help="JSON file for all lines")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_goals.py measures on a CUDA device; none is visible")
    info = gpu_info()
    peak = copy_peak()
    rows = [dict(task="hbm", mode="copy_2GiB", bytes_per_s=peak)]
    print(json.dumps(dict(rows[0], **info)), flush=True)
    for n in a.tabletop_envs:
        for r in bench_tabletop(n, a.rounds, a.min_window, a.calls, peak):
            print(json.dumps(dict(r, **info)), flush=True)
            rows.append(r)
    for task in a.sawyer_tasks:
        for r in bench_sawyer(task, a.sawyer_envs, a.sawyer_steps, a.calls):
            print(json.dumps(dict(r, **info)), flush=True)
            rows.append(r)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"gpu": info, "results": rows}, f, indent=1)


if __name__ == "__main__":
    main()
