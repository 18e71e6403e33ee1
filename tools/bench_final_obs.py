#!/usr/bin/env python
"""What keeping the final observations costs (final_obs=True, EARL_FLAG_FINAL_OBS), one GPU, random actions.

Each configuration builds two auto-reset handles on the same seed, `plain` (auto_reset=True) and `final`
(auto_reset=True, final_obs=True), horizon 64, and steps them on the same action ring, alternating window by window in one
process: every window is a whole number of horizons lasting at least --min-window seconds, timed with CUDA events after one
warm-up horizon per handle, so both handles are always at the same step of the same rollout.  Reports the best window's
env-steps/s of each handle, all windows, and final / plain, with the GPU's name and power limit read in the same run; one
JSON line per configuration, all of them also written to --out.

Configurations: tabletop_manipulation at 1M and 4M envs (fp32 state, sparse), the three-object tabletop at 4M, sawyer_door
and sawyer_peg at 65,536 and kitchen at 14,208 envs -- the sizes the other benchmarks of each task use.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from earl_benchmark_b200.envs import kitchen, sawyer_door, sawyer_peg, tabletop_manipulation  # noqa: E402
from earl_benchmark_b200.envs import tabletop_manipulation_3obj  # noqa: E402
from earl_benchmark_b200.wrappers.persistent_state_wrapper import PersistentStateWrapper  # noqa: E402

HORIZON, RING = 64, 16
CONFIGS = {   # name: (constructor, num_envs, action dim)
    "tabletop_1M": (lambda **k: tabletop_manipulation.TabletopManipulation(reward_type="sparse", **k), 1 << 20, 3),
    "tabletop_4M": (lambda **k: tabletop_manipulation.TabletopManipulation(reward_type="sparse", **k), 4 << 20, 3),
    "tabletop_3obj_4M": (lambda **k: tabletop_manipulation_3obj.TabletopManipulation(reward_type="sparse", **k), 4 << 20, 3),
    "sawyer_door_65536": (lambda **k: sawyer_door.SawyerDoorV2(reward_type="sparse", **k), 65536, 4),
    "sawyer_peg_65536": (lambda **k: sawyer_peg.SawyerPegV2(reward_type="sparse", **k), 65536, 4),
    "kitchen_14208": (lambda **k: kitchen.Kitchen(**k), 14208, 9),
}


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
    except (OSError, subprocess.CalledProcessError):
        name, power = torch.cuda.get_device_name(0), "unknown"
    return {"gpu": name, "power_limit": power}


def run(env, actions, t0, steps):
    for t in range(t0, t0 + steps):
        env.step(actions[t % RING])


def bench(name, rounds, min_window):
    ctor, n, dim = CONFIGS[name]
    g = torch.Generator(device="cuda:0").manual_seed(1234)
    actions = torch.rand((RING, n, dim), generator=g, device="cuda:0") * 2 - 1
    envs = {}
    for mode, extra in (("plain", {}), ("final", {"final_obs": True})):
        envs[mode] = PersistentStateWrapper(ctor(num_envs=n, device="cuda:0", seed=1, auto_reset=True, **extra), HORIZON)
        envs[mode].reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    probe = {}
    for mode, env in envs.items():   # warm-up horizon, then a timed one that sizes the windows
        run(env, actions, 0, HORIZON)
        e0.record()
        run(env, actions, HORIZON, HORIZON)
        e1.record()
        torch.cuda.synchronize()
        probe[mode] = e0.elapsed_time(e1)
    horizons = max(1, int(-(-min_window * 1e3 // min(probe.values()))))
    steps = horizons * HORIZON
    ms = {m: [] for m in envs}
    clock = 2 * HORIZON
    for _ in range(rounds):
        for mode, env in envs.items():
            e0.record()
            run(env, actions, clock, steps)
            e1.record()
            torch.cuda.synchronize()
            ms[mode].append(e0.elapsed_time(e1))
        clock += steps
    rates = {m: [n * steps / (t * 1e-3) for t in ms[m]] for m in envs}
    interv = {m: float(envs[m].num_interventions.double().mean()) for m in envs}
    assert interv["plain"] == interv["final"]   # both handles reset the same envs at the same steps
    row = dict(config=name, num_envs=n, horizon=HORIZON, steps_per_window=steps, windows=rounds,
               env_steps_per_s_plain=max(rates["plain"]), env_steps_per_s_final=max(rates["final"]),
               ratio_final_over_plain=max(rates["final"]) / max(rates["plain"]),
               env_steps_per_s_plain_all=rates["plain"], env_steps_per_s_final_all=rates["final"],
               interventions_per_env=interv["final"])
    for env in envs.values():
        env.env.close()
    del envs, actions
    torch.cuda.empty_cache()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=list(CONFIGS), choices=list(CONFIGS))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--min-window", type=float, default=0.5, help="seconds")
    ap.add_argument("--out", default=None, help="JSON file for all lines")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_final_obs.py measures on a CUDA device; none is visible")
    info = gpu_info()
    rows = []
    for name in a.configs:
        r = bench(name, a.rounds, a.min_window)
        r.update(info)
        print(json.dumps(r), flush=True)
        rows.append(r)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
