#!/usr/bin/env python
"""What the kitchen's evaluation statistics cost, one GPU.

bench.py's kitchen configuration (14,208 envs, seed 0 for the envs, torch.manual_seed(99) random actions, 30 warm-up steps
after a full reset) on two handles in one process: `plain` (no flag) and `eval_stats` (Kitchen(eval_stats=True)).  Both
step the same action sequence from the same state; windows alternate plain, eval_stats, plain, ..., each a whole number of
steps lasting at least --min-window seconds of device time (CUDA events), so both handles stay at the same step of the
rollout in every round.  Then eval_stats() itself: CUDA events around --calls back-to-back calls at each of --stats-envs.
Prints the result as one JSON line and writes it, with the GPU's name and power limit, to OUT/bench_kitchen_eval.json.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from earl_benchmark_b200.envs import kitchen  # noqa: E402

MODES = ("plain", "eval_stats")
WARMUP, RING = 30, 8


def gpu_info():
    """name and power limit of GPU 0 (read-only query)"""
    out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], text=True)
    name, power = [x.strip() for x in out.splitlines()[1].split(",")]
    return {"gpu": name, "power_limit": power}


def make(n, flag):
    env = kitchen.Kitchen(num_envs=n, device="cuda:0", seed=0, eval_stats=flag)
    env.seed(0)
    return env


def timed(fn, count):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(count):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3


def step_cost(n, windows, min_window):
    gen = torch.Generator(device="cuda:0")
    gen.manual_seed(99)
    actions = torch.rand((2 * RING, n, 9), generator=gen, device="cuda:0", dtype=torch.float32) * 2 - 1
    envs = {m: make(n, m == "eval_stats") for m in MODES}
    clock = dict.fromkeys(MODES, 0)

    def run(m, steps):
        t0 = clock[m]
        s = timed(lambda i: envs[m].step(actions[(t0 + i) % RING if t0 + i < WARMUP else RING + (t0 + i) % RING]), steps)
        clock[m] += steps
        return s

    for m in MODES:
        envs[m].reset()
        run(m, WARMUP)
    probe = max(run(m, 2) / 2 for m in MODES)
    steps = max(1, math.ceil(min_window / probe))
    secs = {m: [] for m in MODES}
    for _ in range(windows):
        for m in MODES:
            secs[m].append(run(m, steps))
    rates = {m: [n * steps / s for s in secs[m]] for m in MODES}
    out = {"num_envs": n, "steps_per_window": steps, "windows": windows, "warmup_steps": WARMUP}
    for m in MODES:
        r = rates[m]
        out[m] = {"env_steps_per_s": statistics.median(r), "env_steps_per_s_all": r,
                  "spread": (max(r) - min(r)) / statistics.median(r), "window_s": secs[m]}
    out["ratio_eval_over_plain"] = out["eval_stats"]["env_steps_per_s"] / out["plain"]["env_steps_per_s"]
    out["ratio_per_round"] = [e / p for e, p in zip(rates["eval_stats"], rates["plain"])]
    same = envs["plain"].get_state()["qpos"] == envs["eval_stats"].get_state()["qpos"]
    out["same_final_qpos"] = bool(same.all())
    out["eval_stats"]["stats"] = envs["eval_stats"].eval_stats().tolist()
    return out, envs["eval_stats"]


def reduction_cost(env, calls):
    for _ in range(10):
        env.eval_stats()
    torch.cuda.synchronize()
    s = timed(lambda i: env.eval_stats(), calls)
    return {"num_envs": env.num_envs, "calls": calls, "us_per_call": s / calls * 1e6}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out", help="output directory")
    ap.add_argument("--envs", type=int, default=14208)
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--min-window", type=float, default=0.5, help="seconds of device time per window")
    ap.add_argument("--stats-envs", type=int, nargs="+", default=[14208, 65536])
    ap.add_argument("--calls", type=int, default=100)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_kitchen_eval.py measures on a CUDA device; none is visible")
    res = {"info": gpu_info()}
    res["step"], warm = step_cost(a.envs, a.windows, a.min_window)
    res["eval_stats_call"] = []
    for n in a.stats_envs:
        env = warm if n == warm.num_envs else make(n, True)   # the reduction reads the statistics arrays only: no reset
        res["eval_stats_call"].append(reduction_cost(env, a.calls))
    print(json.dumps(res), flush=True)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_kitchen_eval.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
