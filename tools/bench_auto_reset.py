#!/usr/bin/env python
"""What a reset costs on the articulated-body tasks (sawyer_door, sawyer_peg, kitchen), random actions, one GPU.

Modes, measured in one process and alternated window by window:
  none       no reset: the horizon is never reached
  none+flag  the same with auto_reset=True: what the extra (no-op) reset launch per step costs
  auto       auto_reset=True, horizon 64: envs reset inside step() on the device
  host       horizon 64, host-driven: step, read done.any() back, reset(mask=done)
Every window is a whole number of 64-step horizons lasting at least --min-window seconds, timed with CUDA events after two
warm-up horizons.  All modes step the same action sequence and stay at the same step of it, window by window; without
resets the envs drift into costlier contact regimes as the rollout goes on, so compare modes within a round
(`env_steps_per_s_all[k]`).  Prints one JSON line per task and mode and writes them, with the GPU's name and power limit,
to --out.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from earl_benchmark_b200.envs import kitchen, sawyer_door, sawyer_peg  # noqa: E402
from earl_benchmark_b200.wrappers.persistent_state_wrapper import PersistentStateWrapper  # noqa: E402

HORIZON, NEVER = 64, 1 << 40
MODES = ("none", "none+flag", "auto", "host")


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
    except (OSError, subprocess.CalledProcessError):
        name, power = torch.cuda.get_device_name(0), "unknown"
    return {"gpu": name, "power_limit": power}


def make(task, n, mode):
    horizon = NEVER if mode.startswith("none") else HORIZON
    auto = mode in ("none+flag", "auto")
    if task == "kitchen":
        env = kitchen.Kitchen(num_envs=n, device="cuda:0", seed=1, auto_reset=auto)
    else:
        cls = sawyer_door.SawyerDoorV2 if task == "sawyer_door" else sawyer_peg.SawyerPegV2
        env = cls(reward_type="sparse", num_envs=n, device="cuda:0", seed=1, auto_reset=auto)
    env = PersistentStateWrapper(env, horizon)
    env.reset()
    return env


def run_steps(env, mode, actions, t0, steps):
    ring = actions.shape[0]
    for t in range(t0, t0 + steps):
        _, _, done, _ = env.step(actions[t % ring])
        if mode == "host" and bool(done.any()):
            env.reset(mask=done)


def bench(task, n, rounds, min_window):
    dim = 9 if task == "kitchen" else 4
    g = torch.Generator(device="cuda:0").manual_seed(1234)
    actions = torch.rand((2 * HORIZON, n, dim), generator=g, device="cuda:0") * 2 - 1
    envs = {m: make(task, n, m) for m in MODES}
    clock = {m: 0 for m in MODES}
    for m in MODES:   # warm-up: one horizon, so every mode has reset once
        run_steps(envs[m], m, actions, clock[m], HORIZON)
        clock[m] += HORIZON
    torch.cuda.synchronize()
    # window length: whole horizons lasting at least min_window, sized on a second horizon of every mode (so that all
    # modes stay at the same step of the action sequence and of their rollouts)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    probe = []
    for m in MODES:
        e0.record()
        run_steps(envs[m], m, actions, clock[m], HORIZON)
        e1.record()
        torch.cuda.synchronize()
        clock[m] += HORIZON
        probe.append(e0.elapsed_time(e1))
    horizons = max(1, int(-(-min_window * 1e3 // min(probe))))
    steps = horizons * HORIZON
    ms = {m: [] for m in MODES}
    for _ in range(rounds):
        for m in MODES:
            e0.record()
            run_steps(envs[m], m, actions, clock[m], steps)
            e1.record()
            torch.cuda.synchronize()
            clock[m] += steps
            ms[m].append(e0.elapsed_time(e1))
    out = []
    for m in MODES:
        rates = [n * steps / (t * 1e-3) for t in ms[m]]
        interv = envs[m].num_interventions
        out.append(dict(task=task, mode=m, num_envs=n, horizon=None if m.startswith("none") else HORIZON, steps_per_window=steps,
                        windows=rounds, env_steps_per_s=max(rates), env_steps_per_s_all=rates,
                        launches=int(envs[m].launch_count) if hasattr(envs[m].env, "launch_count") else None,
                        interventions_per_env=float(interv.double().mean())))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tasks", nargs="+", default=["sawyer_door", "sawyer_peg", "kitchen"])
    ap.add_argument("--door-envs", type=int, default=16384)
    ap.add_argument("--kitchen-envs", type=int, default=4096)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--min-window", type=float, default=0.3, help="seconds")
    ap.add_argument("--out", default=None, help="JSON file for all lines")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_auto_reset.py measures on a CUDA device; none is visible")
    info = gpu_info()
    rows = []
    for task in a.tasks:
        n = a.kitchen_envs if task == "kitchen" else a.door_envs
        for r in bench(task, n, a.rounds, a.min_window):
            r.update(info)
            print(json.dumps(r), flush=True)
            rows.append(r)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"gpu": info, "results": rows}, f, indent=1)


if __name__ == "__main__":
    main()
