#!/usr/bin/env python
"""What episode statistics and resets cost on the three-object tabletop, 4,194,304 envs, random actions, one GPU.

Modes, measured in one process and alternated window by window:
  none                the plain step kernel (what bench.py's tabletop_3obj section runs); horizon never reached
  eval                eval_stats=True, horizon never reached: the GENERAL kernel accumulating the episode statistics
  auto                auto_reset=True, horizon 64: envs reset inside the step kernel
  auto+reset_at_goal  the same, every reset taking its qpos from a reset stream of R = 8 rows
  host                horizon 64, host-driven: step, read done.any() back, reset(mask=done)
Every window is a whole number of 64-step horizons lasting at least --min-window seconds, timed with CUDA events after
two warm-up horizons; the state (288 MB) and the per-step traffic are far larger than L2.  Algorithmic bytes per env step:
194 (the plain step) + 16 for the episode return (read + write) + per reset env, amortised over the horizon, 48 for the
object planes the step did not write, 16 for num_interventions and with a stream 64 for the row and 8 for the cursor.
`host` does the same work as `auto` and is charged the same bytes.  Prints one JSON line per mode and writes them, with
the GPU's name and power limit, to --out.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from earl_benchmark_b200.envs.tabletop_manipulation_3obj import TabletopManipulation  # noqa: E402
from earl_benchmark_b200.wrappers.persistent_state_wrapper import PersistentStateWrapper  # noqa: E402

HORIZON, NEVER, ROWS = 64, 1 << 40, 8
MODES = ("none", "eval", "auto", "auto+reset_at_goal", "host")
BASE_BYTES = 194


def bytes_per_env_step(mode):
    extra = {"none": 0.0, "eval": 16.0, "auto": (48 + 16) / HORIZON, "host": (48 + 16) / HORIZON,
             "auto+reset_at_goal": (48 + 16 + 64 + 8) / HORIZON}[mode]
    return BASE_BYTES + extra


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
    except (OSError, subprocess.CalledProcessError):
        name, power = torch.cuda.get_device_name(0), "unknown"
    return {"gpu": name, "power_limit": power}


def make(n, mode):
    kw = dict(reward_type="sparse", num_envs=n, device="cuda:0", seed=1)
    if mode == "eval":
        kw.update(eval_stats=True)
    elif mode == "auto":
        kw.update(auto_reset=True)
    elif mode == "auto+reset_at_goal":
        kw.update(auto_reset=True, reset_at_goal=True, reset_stream_rows=ROWS)
    env = PersistentStateWrapper(TabletopManipulation(**kw), NEVER if mode in ("none", "eval") else HORIZON)
    env.reset()
    return env


def run_steps(env, mode, actions, t0, steps):
    ring = actions.shape[0]
    for t in range(t0, t0 + steps):
        _, _, done, _ = env.step(actions[t % ring])
        if mode == "host" and bool(done.any()):
            env.reset(mask=done)


def bench(n, rounds, min_window):
    g = torch.Generator(device="cuda:0").manual_seed(1234)
    actions = torch.rand((8, n, 3), generator=g, device="cuda:0") * 2 - 1
    envs = {m: make(n, m) for m in MODES}
    clock = {m: 0 for m in MODES}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    probe = []
    for m in MODES:   # warm-up horizon, then a timed one that sizes the windows
        run_steps(envs[m], m, actions, clock[m], HORIZON)
        e0.record()
        run_steps(envs[m], m, actions, clock[m] + HORIZON, HORIZON)
        e1.record()
        torch.cuda.synchronize()
        clock[m] += 2 * HORIZON
        probe.append(e0.elapsed_time(e1))
    steps = max(1, int(-(-min_window * 1e3 // min(probe)))) * HORIZON
    ms = {m: [] for m in MODES}
    launches = {}
    for _ in range(rounds):
        for m in MODES:
            l0 = envs[m].launch_count
            e0.record()
            run_steps(envs[m], m, actions, clock[m], steps)
            e1.record()
            torch.cuda.synchronize()
            launches[m] = envs[m].launch_count - l0
            clock[m] += steps
            ms[m].append(e0.elapsed_time(e1))
    out = []
    for m in MODES:
        best = min(ms[m])
        out.append(dict(mode=m, num_envs=n, horizon=None if m in ("none", "eval") else HORIZON, steps_per_window=steps,
                        windows=rounds, env_steps_per_s=n * steps / (best * 1e-3),
                        env_steps_per_s_all=[n * steps / (t * 1e-3) for t in ms[m]], ms_per_step=best / steps,
                        algorithmic_bytes_per_env_step=bytes_per_env_step(m),
                        algorithmic_gb_per_s=bytes_per_env_step(m) * n * steps / (best * 1e-3) / 1e9,
                        launches_per_step=launches[m] / steps,
                        interventions_per_env=float(envs[m].num_interventions.double().mean())))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4194304)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--min-window", type=float, default=0.3, help="seconds")
    ap.add_argument("--out", default=None, help="JSON file for all lines")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_tt3_features.py measures on a CUDA device; none is visible")
    info = gpu_info()
    rows = []
    for r in bench(a.envs, a.rounds, a.min_window):
        r.update(info)
        print(json.dumps(r), flush=True)
        rows.append(r)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"gpu": info, "results": rows}, f, indent=1)


if __name__ == "__main__":
    main()
