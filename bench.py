#!/usr/bin/env python
"""bench.py -- batched env-steps/sec of the tabletop_manipulation hot path on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--num-envs E] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): tabletop_manipulation, sparse reward, reset-free train horizon
200,000, 1,048,576 envs per GPU (weak scaling), random actions pre-generated on the device
(torch.rand, seed 1234+rank) in a ring of 64 batches (768 MB > L2), observations / rewards / dones
written to a ring of 16 output slots (848 MB > L2).  One "step" = one launch of the fused step kernel
over the whole batch (env.step + PersistentStateWrapper bookkeeping).  `--steps K` is the number of timed
steps: after one untimed K-step priming block, K steps run inside one CUDA-event pair.  e2e times K host-buffer
steps (or --e2e-steps) after three untimed ones; at K = 20 that region is only tens of ms, so a steady e2e figure
wants a larger K.

One JSON line on stdout (rank 0):
  value        whole-job env-steps/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e          same metric through the public API with HOST (pinned) buffers: H2D of the actions and D2H of
               obs/reward/done/success inside the timed region, every step
  roofline     HBM roofline of the step kernel: 113 algorithmic bytes per env-step (SURVEY.md 8d)
  cpu_baseline the CPU oracle (C port of the reference arithmetic, OpenMP, all host threads) on a bounded
               sample of the same workload (rank 0, N=1 only)
  sawyer_door  second section (BASELINE.json configs[2]): batched Sawyer door step, 65,536 envs per GPU, random
               actions; env-steps/s, e2e with host buffers, FP32-issue roofline from the checker's flop count, CPU
               baseline (fp64 C restatement of the engine, one process per host core)
  sawyer_peg   third section (BASELINE.json configs[3]): the same for the Sawyer peg task (free-joint peg, nv = 15)
  kitchen      fourth section (configs[4]): batched Franka kitchen step, 14,208 envs per GPU, 40 substeps per env step
`--impl reference` times that CPU port alone on the same config (the reference itself is Python over
mujoco-py and cannot run on the GPU box; see DESIGN.md).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

ALG_BYTES_PER_ENV_STEP = 113  # SURVEY.md section 8(d): read 36 B, write 77 B
METRIC = "batched env-steps/sec (tabletop_manipulation, sparse, reset-free)"
UNIT = "env-steps/s"
ACTION_RING, OUT_RING = 64, 16
TRAIN_HORIZON = 200000


def measured_peak_gbs():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the benchmark runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,utilization.gpu,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for ts, r in self.rows if (t0 is None or ts >= t0 - 0.1) and (t1 is None or ts <= t1 + 0.1)]
        if not rows:
            rows = [r for _, r in self.rows]
        sm, mx, reasons = [], None, set()
        for r in rows:
            try:
                clk, mxc, util = float(r[0]), float(r[1]), float(r[3])
            except Exception:
                continue
            mx = mxc
            if util >= 10:
                sm.append(clk)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(rows)}


# ----------------------------------------------------------------------------------------------- CPU arm

def cpu_port_rate(num_envs, steps, threads, budget_s=20.0, min_wall_s=0.0):
    """env-steps/s of the CPU oracle (step-major: all envs advance one step at a time, like a vector env).
    The sample is bounded to about `budget_s` seconds: fewer envs per step if needed, never fewer steps."""
    import numpy as np
    os.environ["OMP_NUM_THREADS"] = str(threads)
    from oracle import loader
    L = loader.lib()
    ring = 4

    def run(n, k):
        rs = np.random.RandomState(1234)
        acts = rs.uniform(-1, 1, (ring, n, 3)).astype(np.float32)
        qpos = np.tile(np.array([0.0, 0.0, 2.5, 0.0]), (n, 1))
        att = np.zeros(n, np.int32)
        goal = np.tile(loader.INITIAL_STATE, (n, 1))
        goal[:, 2:4] = loader.GOAL_STATES[rs.randint(0, 4, n), 2:4]
        total, since = np.zeros(n, np.int64), np.zeros(n, np.int64)
        obs, rew, done = np.zeros((n, 12), np.float32), np.zeros(n), np.zeros(n, np.uint8)
        t0 = time.perf_counter()
        L.earl_oracle_tt_rollout_stepmajor(n, k, ring, qpos, att, goal, acts, 0, 0, 1, total, since, TRAIN_HORIZON,
                                           obs, rew, done)
        return time.perf_counter() - t0

    n = min(num_envs, 1 << 16)
    run(n, 2)                      # touch pages, spin up threads
    t = run(n, 8) / 8              # seconds per step at the calibration size
    per_env_step = t / n
    n_sample = num_envs
    if per_env_step * num_envs * steps > budget_s:
        n_sample = max(1 << 14, int(budget_s / (per_env_step * steps)))
        n_sample = min(num_envs, n_sample)
    # a sample worth timing: at least `min_wall_s` seconds on all threads (tens of core-seconds), by more steps of the same batch
    k = max(steps, int(min_wall_s / max(per_env_step * n_sample, 1e-9)) + 1)
    el = run(n_sample, k)
    return n_sample * k / el, n_sample, el, k


# ----------------------------------------------------------------------------------------------- Sawyer door (config 3)

DOOR_ENVS, DOOR_STEPS, DOOR_WARMUP, DOOR_RING = 1 << 16, 100, 100, 16
DOOR_FRESH_STEPS, DOOR_FRESH_WARMUP = 30, 5


def door_cpu_rate(procs, steps_per_proc=20000, task="sawyer_door"):
    """env-steps/s of the fp64 checker on `procs` host processes (oracle/door_cpu_bench.py, one checker instance each:
    oracle/mjengine.c keeps static scratch, so it is not thread-safe), and its flop count per env step -- the
    ALGORITHMIC flops of SURVEY.md 8d, counted inside the checker on the same random-action workload."""
    script = os.path.join(REPO, "oracle", "door_cpu_bench.py")
    env = dict(os.environ, OMP_NUM_THREADS="1")
    subprocess.check_call([sys.executable, script, "0", "5", task], stdout=subprocess.DEVNULL, env=env)  # builds the checker once
    t0 = time.perf_counter()
    ps = [subprocess.Popen([sys.executable, script, str(100 + k), str(steps_per_proc), task], stdout=subprocess.PIPE, text=True, env=env)
          for k in range(procs)]
    res = [json.loads(p.communicate()[0].strip().splitlines()[-1]) for p in ps]
    wall = time.perf_counter() - t0
    loop = max(r["seconds"] for r in res)
    flops = sum(r["flops_per_env_step"] for r in res) / len(res)
    return procs * steps_per_proc / loop, flops, wall



def host_path_note():
    """Which of earl_step_host's two data paths this process uses (earl_set_host_zerocopy, envs/_hostio.py)."""
    from earl_benchmark_b200.envs import _hostio
    zc = _hostio.host_zerocopy_default()
    if zc is None:
        zc = int(os.environ.get("EARL_TT_HOST_ZEROCOPY", "1") != "0")
    return ("the step kernel reads / writes the pinned host buffers over PCIe itself, one launch per step" if zc else
            "staged pipeline of host->device copy, kernel, device->host copies (several ranks share this host)")


ENGINE_CAPTURES = {
    "sawyer_door": ("prof_door_steady_16k_r02.raw.csv", "sawyer_door, 16,384 envs, steady regime, serial-redo build of round 2"),
    "sawyer_peg": ("prof_peg_steady_16k_final.raw.csv", "sawyer_peg, 16,384 envs, env step 105 of the rollout, final build of round 2"),
    "kitchen": ("prof_kitchen_steady_4736_r02.raw.csv", "kitchen, 4,736 envs, env step 32 of the rollout, two barrier domains"),
}


def ncu_engine_summary(task="sawyer_door"):
    """A few figures of the committed `ncu --set full` capture of the step kernel on this task (profiles/r02/, ENGINE_CAPTURES)
    -- read from the file, never typed in; None when the file is not there."""
    import csv
    fname, what = ENGINE_CAPTURES[task]
    path = os.path.join(REPO, "profiles", "r02", fname)
    try:
        rows = list(csv.reader(open(path)))
        hdr, val = rows[0], rows[2]
        g = lambda k: float(val[hdr.index(k)].replace(",", ""))  # noqa: E731
        return {"source": f"profiles/r02/{fname} ({what}; not this run)",
                "executed_ipc": g("sm__inst_executed.avg.per_cycle_active"),
                "achieved_occupancy_pct": g("sm__warps_active.avg.pct_of_peak_sustained_active"),
                "issue_slots_busy_pct": g("smsp__issue_active.avg.pct_of_peak_sustained_active"),
                "active_lanes_per_instruction": g("smsp__thread_inst_executed_per_inst_executed.ratio"),
                "registers_per_thread": g("launch__registers_per_thread"), "kernel_ms": g("gpu__time_duration.sum")}
    except Exception:
        return None


def run_door(dev, rank, world, sm_max_mhz, sm_count, with_cpu, task="sawyer_door"):
    """Second / third bench section: batched sawyer_door (BASELINE.json configs[2]) or sawyer_peg (configs[3]) step,
    65,536 envs per GPU, random actions."""
    import torch
    import torch.distributed as dist

    from earl_benchmark_b200.distributed import max_over_ranks
    from earl_benchmark_b200.envs import sawyer_door, sawyer_peg

    n = DOOR_ENVS
    door = task == "sawyer_door"
    env = (sawyer_door.SawyerDoorV2 if door else sawyer_peg.SawyerPegV2)(reward_type="sparse", num_envs=n, device=dev, seed=rank)
    env.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(4321 + rank)
    actions = torch.rand((DOOR_RING, n, 4), generator=gen, device=dev, dtype=torch.float32) * 2 - 1
    # (a) right after the reset: arms settled, grippers open, nobody touches the door yet
    for t in range(DOOR_FRESH_WARMUP):
        env.step(actions[t % DOOR_RING])
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for t in range(DOOR_FRESH_STEPS):
        env.step(actions[(DOOR_FRESH_WARMUP + t) % DOOR_RING])
    f1.record()
    torch.cuda.synchronize()
    ms_fresh = max_over_ranks(f0.elapsed_time(f1), dev)
    # (b) the judged window: DOOR_WARMUP steps into the random rollout, when a steady share of the grippers is on the
    # handle / the table (more contacts, more Newton iterations); this is the number reported as `value`
    for t in range(DOOR_FRESH_WARMUP + DOOR_FRESH_STEPS, DOOR_WARMUP):
        env.step(actions[t % DOOR_RING])
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    w0 = env.work_counters()
    l0 = env.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(DOOR_STEPS):
        env.step(actions[t % DOOR_RING])
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1), dev)
    w1 = env.work_counters()
    launches = env.launch_count - l0
    # end to end with host buffers
    host_a = (torch.rand((n, 4), dtype=torch.float32) * 2 - 1).pin_memory()
    env.step(host_a)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        env.step(host_a)
    e2e_s = max_over_ranks(time.perf_counter() - t0, dev)
    out = None
    if rank == 0:
        sub = max(1, w1["substeps"] - w0["substeps"])
        value = n * world * DOOR_STEPS / (ms * 1e-3)
        out = {"metric": f"batched env-steps/sec ({task}, sparse, 5 substeps per env step)", "value": value, "unit": UNIT,
               "envs_per_gpu": n, "steps": DOOR_STEPS, "warmup": DOOR_WARMUP, "ms_per_step": ms / DOOR_STEPS,
               "dtype": "f32", "gpu_launches": launches,
               "window": f"steps {DOOR_WARMUP}..{DOOR_WARMUP + DOOR_STEPS} of a random-action rollout after reset",
               "first_steps_after_reset": {"value": n * world * DOOR_FRESH_STEPS / (ms_fresh * 1e-3), "unit": UNIT,
                                           "steps": DOOR_FRESH_STEPS, "warmup": DOOR_FRESH_WARMUP,
                                           "note": "lighter workload: only the four door-on-table contacts per env" if door else
                                                   "peg lying on the table, gripper above it"},
               "e2e": {"value": n * world * 5 / e2e_s, "unit": UNIT, "h2d_bytes_per_step": n * 16 * world,
                       "d2h_bytes_per_step": n * (14 * 4 + 4 + 1 + 1) * world, "steps": 5},
               "work": {"newton_iterations_per_substep": (w1["newton_iterations"] - w0["newton_iterations"]) / sub,
                        "constraint_rows_per_substep": (w1["constraint_rows"] - w0["constraint_rows"]) / sub,
                        "contacts_per_substep": (w1["contacts"] - w0["contacts"]) / sub,
                        "bad_states": w1["bad_states"] - w0["bad_states"],
                        "overflow_states": w1["overflow_states"] - w0["overflow_states"]},
               "kernel": "mj_step_kernel (one warp per env, 16 envs per SM in flight, small capacity set) + concurrent mj_redo_kernel "
                         "(extra-large capacity set, re-steps capacity overflows) + mj_order_kernel (visiting order, <4 us)",
               "redone_states": w1.get("redone_states", 0) - w0.get("redone_states", 0),
               "ncu": ncu_engine_summary(task)}
        if with_cpu:
            procs = os.cpu_count() or 1
            rate, flops, wall = door_cpu_rate(procs, task=task)
            peak = sm_count * 128 * 2 * (sm_max_mhz or 1965.0) * 1e6 / 1e12
            ach = flops * (value / world) / 1e12
            out["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": procs, "kind": "port",
                                   "sample": f"{procs} processes x 20000 env steps of the same random-action workload, fp64 "
                                             f"C restatement of the engine (not MuJoCo), {wall:.1f} s"}
            out["roofline"] = {"bound": "fp32", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                               "traffic": None, "algorithmic_flops_per_env_step": flops,
                               "peak_source": f"{sm_count} SMs x 128 lanes x 2 x {sm_max_mhz or 1965.0:.0f} MHz (nominal FP32 FMA issue)",
                               "note": "algorithmic flops = the checker's own flop counter on the same workload; the kernel is "
                                       "latency / instruction-issue bound on per-env serial chains, not FMA bound"}
    del env
    return out


KITCHEN_ENVS, KITCHEN_STEPS, KITCHEN_WARMUP = 14208, 8, 30


def run_kitchen(dev, rank, world, sm_max_mhz, sm_count, with_cpu):
    """Fourth bench section: batched kitchen step (BASELINE.json configs[4]): 14,208 envs per GPU (= 148 SMs x 8 resident
    environments x 12 waves), random actions after a full reset (400 settle substeps per env)."""
    import torch
    import torch.distributed as dist

    from earl_benchmark_b200.distributed import max_over_ranks
    from earl_benchmark_b200.envs import kitchen

    n = KITCHEN_ENVS
    env = kitchen.Kitchen(num_envs=n, device=dev, seed=1000 * rank)
    env.seed(1000 * rank)
    env.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(99 + rank)
    actions = torch.rand((8 + KITCHEN_STEPS, n, 9), generator=gen, device=dev, dtype=torch.float32) * 2 - 1
    for t in range(KITCHEN_WARMUP):
        env.step(actions[t % 8])
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    w0 = env.work_counters()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(KITCHEN_STEPS):
        env.step(actions[8 + t])
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1), dev)
    w1 = env.work_counters()
    host_a = (torch.rand((n, 9), dtype=torch.float32) * 2 - 1).numpy()
    t0 = time.perf_counter()
    for _ in range(2):
        env.step(host_a)
    e2e_s = max_over_ranks(time.perf_counter() - t0, dev)
    out = None
    if rank == 0:
        sub = max(1, w1["substeps"] - w0["substeps"])
        value = n * world * KITCHEN_STEPS / (ms * 1e-3)
        out = {"metric": "batched env-steps/sec (kitchen, dense, 40 substeps per env step)", "value": value, "unit": UNIT,
               "envs_per_gpu": n, "steps": KITCHEN_STEPS, "warmup": KITCHEN_WARMUP, "ms_per_step": ms / KITCHEN_STEPS, "dtype": "f32",
               "gpu_launches": 4 * KITCHEN_STEPS,   # task kernel + redo kernel + two tiny kernels that build the next visiting order
               "window": f"env steps {KITCHEN_WARMUP}..{KITCHEN_WARMUP + KITCHEN_STEPS} of a random-action rollout after a full reset "
                         "(arms up to speed: the broad-phase cache is rebuilt more often than right after the reset)",
               "e2e": {"value": n * world * 2 / e2e_s, "unit": UNIT, "h2d_bytes_per_step": n * 36 * world,
                       "d2h_bytes_per_step": n * (46 * 8 + 8 + 1 + 1) * world, "steps": 2},
               "work": {"newton_iterations_per_substep": (w1["newton_iterations"] - w0["newton_iterations"]) / sub,
                        "constraint_rows_per_substep": (w1["constraint_rows"] - w0["constraint_rows"]) / sub,
                        "contacts_per_substep": (w1["contacts"] - w0["contacts"]) / sub,
                        "bad_states": w1["bad_states"] - w0["bad_states"],
                        "overflow_states": w1["overflow_states"] - w0["overflow_states"],
                        "redone_states": w1["redone_states"] - w0["redone_states"]},
               "kernel": "mjk_task_kernel (one warp per env, 8 envs per SM in flight, 112-row workspaces, model tables in global memory, cost-sorted visiting order, dynamic chunks) "
                         "+ mjk_redo_kernel (544-row set, concurrent on four reserved SMs plus every SM the step kernel vacates: the ~0.1 % of env steps that outgrew 112 rows / 24 contacts)",
               "ncu": ncu_engine_summary("kitchen")}
        if with_cpu:
            procs = os.cpu_count() or 1
            rate, flops, wall = door_cpu_rate(procs, steps_per_proc=1500, task="kitchen")
            peak = sm_count * 128 * 2 * (sm_max_mhz or 1965.0) * 1e6 / 1e12
            ach = flops * (value / world) / 1e12
            out["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": procs, "kind": "port",
                                   "sample": f"{procs} processes x 1500 env steps of the same random-action workload, fp64 C "
                                             f"restatement of the engine + pinned task logic (not MuJoCo), {wall:.1f} s"}
            out["roofline"] = {"bound": "fp32", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                               "algorithmic_flops_per_env_step": flops,
                               "peak_source": f"{sm_count} SMs x 128 lanes x 2 x {sm_max_mhz or 1965.0:.0f} MHz (nominal FP32 FMA issue)",
                               "note": "8 warps per SM (27 KB workspace and 246 registers per env both bind there), cached broad phase, "
                                       "cost-sorted dynamic chunks; bound by per-warp dependent latency and the phase barriers, not by FMA issue"}
    del env
    return out


TT3_ENVS = 1 << 22           # per GPU: 288 MB of state, so state, actions and outputs all stream from HBM
TT3_ALG_BYTES = 194           # read action 12 + qpos 64 + meta 8; write fist 16 + meta 8 + obs 80 + reward 4 + done 1
                              # + success 1 (+ 16 for the dragged object of the envs that hold one: not counted)


def run_tt3(dev, rank, world, with_e2e):
    """Three-object tabletop section (reference envs/tabletop_manipulation_3obj.py; SURVEY 8(f) row 4): batched step at
    4,194,304 envs per GPU, random actions, sparse reward, reset-free horizon never reached."""
    import torch
    import torch.distributed as dist

    from earl_benchmark_b200.distributed import max_over_ranks
    from earl_benchmark_b200.envs.tabletop_manipulation_3obj import TabletopManipulation
    from earl_benchmark_b200.wrappers.persistent_state_wrapper import PersistentStateWrapper

    n, warm, steps = TT3_ENVS, 20, 200
    env = PersistentStateWrapper(TabletopManipulation(reward_type="sparse", num_envs=n, device=dev, seed=rank), TRAIN_HORIZON)
    env.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(977 + rank)
    actions = torch.rand((8, n, 3), generator=gen, device=dev, dtype=torch.float32) * 2 - 1
    obs = torch.empty((4, n, 20), device=dev, dtype=torch.float32)
    rew = torch.empty((4, n), device=dev, dtype=torch.float32)
    done = torch.empty((4, n), device=dev, dtype=torch.uint8)
    succ = torch.empty((4, n), device=dev, dtype=torch.uint8)
    env.rollout_into(actions, warm, obs, rew, done, succ)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = env.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    env.rollout_into(actions, steps, obs, rew, done, succ)
    e1.record()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1), dev)
    _, att = env.get_state()
    out = {"workload": "tabletop_manipulation_3obj sparse reward, reset-free, random actions", "envs_per_gpu": n, "steps": steps,
           "warmup": warm, "value": n * world * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps,
           "gpu_launches": env.launch_count - l0, "kernel": "tt3_step_kernel (one thread per env, shared-memory tiles, PDL)",
           "algorithmic_bytes_per_env_step": TT3_ALG_BYTES,
           "achieved": TT3_ALG_BYTES * n / (ms * 1e-3 / steps) / 1e9,
           "holding_fraction": float((att > 0).float().mean()),
           "l2": "inputs larger than L2: state 288 MB, action ring 8 x 50 MB, output ring 4 x 360 MB"}
    if with_e2e:
        # CPU baseline of this section: the numpy restatement (oracle/tabletop3.py) on one host core, bounded sample
        from oracle.tabletop3 import Tabletop3Oracle
        cn, ck = 1 << 16, 100
        orc = Tabletop3Oracle(cn, TRAIN_HORIZON)
        orc.reset()
        ca = actions[0, :cn].cpu().numpy()
        orc.step(ca)
        c0 = time.perf_counter()
        for _ in range(ck):
            orc.step(ca)
        cel = time.perf_counter() - c0
        out["cpu_baseline"] = {"value": cn * ck / cel, "unit": UNIT, "cores": 1, "kind": "port",
                               "sample": f"{cn} envs x {ck} steps, vectorised numpy restatement of the reference class, {cel:.2f} s"}
        m = 1 << 20
        del env, obs, rew, done, succ, actions
        e = PersistentStateWrapper(TabletopManipulation(reward_type="sparse", num_envs=m, device=dev, seed=rank), TRAIN_HORIZON)
        e.reset()
        ha = [torch.rand((m, 3), dtype=torch.float32).mul_(2).sub_(1).pin_memory() for _ in range(4)]
        for t in range(3):
            e.step(ha[t % 4])
        t0 = time.perf_counter()
        k = 20
        for t in range(k):
            e.step(ha[t % 4])
        el = time.perf_counter() - t0
        out["e2e"] = {"value": m * k / el, "unit": UNIT, "envs": m, "steps": k, "h2d_bytes_per_step": m * 12,
                      "d2h_bytes_per_step": m * (80 + 4 + 1 + 1),
                      "api": "PersistentStateWrapper.step(pinned host actions) -> host obs/reward/done/success"}
    return out


def ref_python_loop():
    """The UNMODIFIED reference's own Python step loop (SURVEY 8(d) CPU baseline (i)), measured where /root/reference exists
    (oracle/ref_python_rate.py, build container) and committed: the GPU box cannot run it."""
    p = os.path.join(REPO, "profiles", "r02", "ref_python_loop_rate.json")
    try:
        d = json.load(open(p))
        return {"unit": UNIT, "measured_in": "build container (8 host cpus), committed as profiles/r02/ref_python_loop_rate.json",
                "runs": [{"procs": r["procs"], "value": r["env_steps_per_s"]} for r in d["runs"]]}
    except Exception:
        return None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    n_total = args.num_envs * args.gpus
    cpu_port_rate(1 << 14, max(1, args.warmup), threads, budget_s=2.0)
    rate, n_sample, el, k = cpu_port_rate(n_total, args.steps, threads, budget_s=90.0, min_wall_s=1.5)
    sample = (f"{n_sample} of {n_total} envs x {k} steps, step-major, OpenMP {threads} threads, "
              f"{el:.2f} s; C port of reference tabletop step + PersistentStateWrapper (the reference itself is Python "
              "over mujoco-py and cannot run here)")
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * n_total / rate, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(args, n_total),
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                             "reference_python_loop": ref_python_loop()},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


def config_dict(args, n_total):
    return {"workload": "tabletop_manipulation sparse reward, reset-free train horizon 200000, random actions "
                        "(BASELINE.json configs[1])",
            "envs_per_gpu": args.num_envs, "total_envs": n_total, "state_dtype": "float32",
            "action_ring": ACTION_RING, "out_ring": OUT_RING,
            "l2": "inputs larger than L2: action ring 64 x 12.6 MB, output ring 16 x 55.6 MB; per-env state "
                  "(25 MB) is deliberately left L2-resident between steps",
            "parallelism": f"env-sharded x{args.gpus}, no collective on the step path"}


# ----------------------------------------------------------------------------------------------- GPU arm

MIN_REGION_S = 0.30      # a sweep point repeats its K-step block until the CUDA-event pair brackets this much device time
DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this many bytes in all, .npy headers included
NPY_HEADER_BYTES = 4096  # bound on the header numpy writes in front of one .npy array


def pin_to_gpu_numa(local):
    """Run this rank on the CPUs NVML reports as local to its GPU BEFORE any pinned allocation, so that first-touch puts
    the pinned staging buffers on the GPU's own NUMA node (matters when 8 ranks share the host)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
        return f"{len(cpus)} cpus [{min(cpus)}..{max(cpus)}]" if cpus else "nvml affinity empty"
    except Exception as e:  # not fatal: the default placement is what round 1 measured
        return f"unavailable ({type(e).__name__})"


def timed_blocks(rollout, steps, barrier, dev, reps=None):
    """Time R repetitions of the K-step block with ONE CUDA-event pair on the launching stream.

    barrier -> one untimed K-step priming block (the NCCL barrier kernel evicts the L2-resident state and the first
    launches after it pay for that; at N=1 it is a no-op) -> [reps None: estimate the block time -> choose R so the timed
    region is >= MIN_REGION_S (same R on every rank) -> barrier -> priming block] -> e0, R x K steps, e1 -> sync -> max
    over ranks.  Returns (ms_total, reps)."""
    import torch

    from earl_benchmark_b200.distributed import max_over_ranks
    barrier()
    rollout(steps)
    if reps is None:
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        rollout(steps)
        a1.record()
        torch.cuda.synchronize()
        est_ms = max(max_over_ranks(a0.elapsed_time(a1), dev), 1e-3)
        reps = int(min(4096, max(1, -(-MIN_REGION_S * 1e3 // est_ms))))
        barrier()
        rollout(steps)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        rollout(steps)
    e1.record()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1), dev)
    barrier()
    return ms, reps


def tabletop_point(eb, dev, rank, world, barrier, n, steps, gen, label, alg_bytes=ALG_BYTES_PER_ENV_STEP, **kw):
    """One extra operating point of the tabletop step (SURVEY 8(d) config 2): n envs per GPU, `steps`-step blocks."""
    import torch
    ring_a, ring_o = (64, 16) if n <= (1 << 20) else (8, 4)
    loader = eb.EARLEnvs("tabletop_manipulation", reward_type="sparse", num_envs=n * world, rank=rank, world_size=world,
                         device=dev, seed=0, goal_stream_rows=kw.pop("goal_stream_rows", 2), **kw)
    train, _ = loader.get_envs()
    train.reset()
    a = torch.rand((ring_a, n, 3), generator=gen, device=dev, dtype=torch.float32) * 2 - 1
    o = torch.empty((ring_o, n, 12), device=dev, dtype=torch.float32)
    r = torch.empty((ring_o, n), device=dev, dtype=torch.float32)
    d = torch.empty((ring_o, n), device=dev, dtype=torch.uint8)
    env = train.env
    env.rollout_into(a, 20, o, r, d)
    l0 = env.launch_count
    ms, reps = timed_blocks(lambda k: env.rollout_into(a, k, o, r, d), steps, barrier, dev)
    per_launch_s = ms * 1e-3 / (steps * reps)
    out = {"point": label, "envs_per_gpu": n, "total_envs": n * world, "steps": steps, "reps": reps,
           "value": n * world / per_launch_s, "unit": UNIT, "ms_per_step": per_launch_s * 1e3,
           "achieved": alg_bytes * n / per_launch_s / 1e9, "algorithmic_bytes_per_env_step": alg_bytes,
           "num_interventions_mean": float(train.num_interventions.double().mean()) if hasattr(train.num_interventions, "double") else None}
    del a, o, r, d, train, loader, env
    torch.cuda.empty_cache()
    return out


def pcie_ceiling(dev, n, barrier, reps=10):
    """The e2e roofline: this step's own byte mix (12 B up, 54 B down per env) moved with plain pinned cudaMemcpyAsync on
    two streams, all ranks at once -- no kernel, no library of this repo involved."""
    import torch

    from earl_benchmark_b200.distributed import max_over_ranks
    up = torch.empty((n, 3), dtype=torch.float32).pin_memory()
    down = [torch.empty((n, 12), dtype=torch.float32).pin_memory(), torch.empty((n,), dtype=torch.float32).pin_memory(),
            torch.empty((n, 2), dtype=torch.uint8).pin_memory()]
    d_up = torch.empty((n, 3), dtype=torch.float32, device=dev)
    d_down = [torch.empty_like(t, device=dev) for t in down]
    s_up, s_down = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def once():
        with torch.cuda.stream(s_up):
            d_up.copy_(up, non_blocking=True)
        with torch.cuda.stream(s_down):
            for h, g in zip(down, d_down):
                h.copy_(g, non_blocking=True)
    once()
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    torch.cuda.synchronize()
    el = max_over_ranks(time.perf_counter() - t0, dev)
    return n * reps / el, (n * 54 * reps) / el / 1e9, (n * 12 * reps) / el / 1e9


def eval_collective_check(eb, dev, rank, world, barrier):
    """SURVEY 8(e): the system's ONE collective, on hardware.  Every rank runs a short evaluation episode on its shard of the
    eval env, reduces (sum return, successes, N) on the device, and all-reduces the 4 doubles over NCCL; the result must
    equal the sum of the per-rank vectors gathered separately, and count every env of the job."""
    import torch
    import torch.distributed as dist

    from earl_benchmark_b200.distributed import all_reduce_eval_stats
    n = 4096
    loader = eb.EARLEnvs("tabletop_manipulation", reward_type="sparse", num_envs=n * world, rank=rank, world_size=world,
                         device=dev, seed=0, eval_horizon=50)
    _, ev = loader.get_envs()
    ev.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(555 + rank)
    for _ in range(50):
        ev.step(torch.rand((n, 3), generator=gen, device=dev) * 2 - 1)
    local = ev.env.eval_stats().clone()
    gathered = [torch.zeros_like(local) for _ in range(world)]
    if world > 1:
        dist.all_gather(gathered, local)
    else:
        gathered = [local]
    expect = torch.stack(gathered).sum(0)
    barrier()
    red = local.clone()
    lat = []
    for k in range(12):     # first calls include NCCL's lazy channel setup: report the steady latency
        buf = local.clone()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        stats = all_reduce_eval_stats(buf)
        lat.append(time.perf_counter() - t0)
        red = buf
    ok = bool(torch.equal(red, expect)) and stats["num_envs"] == n * world
    if not ok:
        raise SystemExit(f"eval all-reduce mismatch: {red.tolist()} vs {expect.tolist()}, num_envs {stats['num_envs']}")
    return {"world_size": world, "backend": "nccl" if world > 1 else "none (single process)", "num_envs": stats["num_envs"],
            "mean_return": stats["mean_return"], "success_rate": stats["success_rate"],
            "equals_sum_of_gathered_per_rank_stats": ok, "latency_us_median": 1e6 * statistics.median(lat[2:]),
            "latency_us_first": 1e6 * lat[0], "bytes": 32}


def ncu_traffic(num_envs):
    """dram bytes per launch of the dominant kernel at this batch size, from the committed `ncu --set full` captures
    (profiles/ncu_traffic.json, keyed by envs per GPU); None when no capture exists for the configuration."""
    try:
        t = json.load(open(os.path.join(REPO, "profiles", "ncu_traffic.json")))["tabletop"].get(str(num_envs))
        return (t["dram_bytes_read"] + t["dram_bytes_write"], t["source"]) if t else (None, None)
    except Exception:
        return None, None


def dump_outputs(out_dir, outputs):
    """Write the device tensors `outputs` (name -> [N, ...], one row per env) as out_dir/<name>.npy in float32.  When they
    would exceed DUMP_BYTES, the same seeded sample of rows is written for every tensor, its env indices as
    env_index.npy (float64)."""
    import numpy as np
    import torch
    n = next(iter(outputs.values())).shape[0]
    row_bytes = sum(4 * t[0].numel() for t in outputs.values())
    payload = DUMP_BYTES - NPY_HEADER_BYTES * (len(outputs) + 1)
    idx = None
    if n * row_bytes > payload:
        idx = np.sort(np.random.RandomState(0).choice(n, payload // (row_bytes + 8), replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        if idx is not None:
            t = t[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
    if idx is not None:
        np.save(os.path.join(out_dir, "env_index.npy"), idx.astype(np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist

    import earl_benchmark_b200 as eb
    from earl_benchmark_b200.distributed import init_from_env, max_over_ranks

    rank, world, local = init_from_env()
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    numa = pin_to_gpu_numa(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    n = args.num_envs
    n_total = n * world

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    loader = eb.EARLEnvs("tabletop_manipulation", reward_type="sparse", num_envs=n_total, rank=rank, world_size=world,
                         device=dev, seed=0, train_horizon=TRAIN_HORIZON, goal_stream_rows=2)
    train, _ = loader.get_envs()
    train.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    actions = torch.rand((ACTION_RING, n, 3), generator=gen, device=dev, dtype=torch.float32) * 2 - 1
    obs = torch.empty((OUT_RING, n, 12), device=dev, dtype=torch.float32)
    rew = torch.empty((OUT_RING, n), device=dev, dtype=torch.float32)
    done = torch.empty((OUT_RING, n), device=dev, dtype=torch.uint8)
    env = train.env
    sampler = ClockSampler(local) if rank == 0 else None

    # warm-up: W steps as asked, then keep the GPU busy for >= 1 s so clocks are sampled under load; that second part runs a
    # time-dependent number of steps, so the state is put back to where the W steps left it: with the same arguments the
    # timed steps see the same inputs in every run
    env.rollout_into(actions, max(args.warmup, 3), obs, rew, done)
    warm_state = env.get_state()
    t_w = time.perf_counter()
    while not args.profile and time.perf_counter() - t_w < 1.0:
        env.rollout_into(actions, 256, obs, rew, done)
        torch.cuda.synchronize()
    env.set_state(warm_state)
    del warm_state

    # ---- device-resident timing: the K timed steps inside one CUDA-event pair
    launches0 = env.launch_count
    t_region0 = time.perf_counter()
    if args.profile:
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        env.rollout_into(actions, args.steps, obs, rew, done)
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1), dev)
        launches = env.launch_count - launches0
    else:
        ms, _ = timed_blocks(lambda k: env.rollout_into(actions, k, obs, rew, done), args.steps, barrier, dev, reps=1)
        launches = env.launch_count - launches0 - args.steps   # the K-step priming block is outside the region
    t_region1 = time.perf_counter()
    per_launch_s = ms * 1e-3 / args.steps
    value = n_total / per_launch_s
    if args.dump_outputs and rank == 0:
        last = (args.steps - 1) % OUT_RING
        dump_outputs(args.dump_outputs, {"obs": obs[last], "reward": rew[last], "done": done[last]})

    # ---- end to end through the public API with host buffers
    e2e_steps = args.steps if args.e2e_steps is None else args.e2e_steps
    if args.profile:
        e2e_steps = 1
    host_actions = [(torch.rand((n, 3), dtype=torch.float32) * 2 - 1).pin_memory() for _ in range(4)]
    for k in range(3):
        train.step(host_actions[k % 4])
    barrier()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        ho, hr, hd, hinfo = train.step(host_actions[k % 4])   # numpy views of pinned result buffers
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0, dev)
    e2e_value = n_total * e2e_steps / e2e_s
    h2d = n * 3 * 4
    d2h = n * (12 * 4 + 4 + 1 + 1)
    ceiling = None
    if not args.profile:
        c_rate, c_down, c_up = pcie_ceiling(dev, n, barrier)
        ceiling = {"value": c_rate * world, "unit": UNIT, "d2h_gbs_per_gpu": c_down, "h2d_gbs_per_gpu": c_up,
                   "how": "the step's own byte mix (12 B up + 54 B down per env) as plain pinned cudaMemcpyAsync on two streams, "
                          f"all {world} ranks concurrently, no kernel; pinned buffers allocated after binding to the GPU's NUMA "
                          f"cpus ({numa})"}
    clocks = sampler.stop(t_region0, t_region1) if sampler else None

    # ---- SURVEY 8(d) config 2: the other batch sizes, strong scaling, the done / auto-reset path, fp64 state, all-HBM points
    sweep, big = [], None
    if not args.profile and not args.no_hbm_check:
        del actions, obs, rew, done
        torch.cuda.empty_cache()
        k = max(20, min(args.steps, 200))
        pts = [("weak 65,536 envs per GPU", 1 << 16, {}, ALG_BYTES_PER_ENV_STEP),
               ("weak 262,144 envs per GPU", 1 << 18, {}, ALG_BYTES_PER_ENV_STEP),
               ("strong 1,048,576 envs in total", (1 << 20) // world, {}, ALG_BYTES_PER_ENV_STEP),
               ("train_horizon=64 with auto_reset (done fires every 64 steps, reset + goal draw inside the step kernel)",
                1 << 20, dict(train_horizon=64, auto_reset=True, goal_stream_rows=64), ALG_BYTES_PER_ENV_STEP),
               ("state_dtype=float64 (the bit-exact operating point: fp64 qpos, 32 B r + 32 B w instead of 16 + 16)",
                1 << 20, dict(state_dtype="float64", train_horizon=TRAIN_HORIZON), ALG_BYTES_PER_ENV_STEP + 32),
               ("all-HBM 4,194,304 envs per GPU (one-tile-per-CTA kernel)", 1 << 22, dict(train_horizon=TRAIN_HORIZON), ALG_BYTES_PER_ENV_STEP),
               ("all-HBM 8,388,608 envs per GPU (one-tile-per-CTA kernel)", 1 << 23, dict(train_horizon=TRAIN_HORIZON), ALG_BYTES_PER_ENV_STEP)]
        for label, npg, kw, ab in pts:
            kw.setdefault("train_horizon", TRAIN_HORIZON)
            sweep.append(tabletop_point(eb, dev, rank, world, barrier, npg, k, gen, label, alg_bytes=ab, **kw))
        big = dict(sweep[-1], kernel="earl::tabletop_step_tile_kernel (one 256-env tile per CTA, PDL)")
    collective = eval_collective_check(eb, dev, rank, world, barrier) if not args.profile else None

    door = peg = kit = tt3 = None
    if not args.profile and not args.no_door:
        props = torch.cuda.get_device_properties(dev)
        tt3 = run_tt3(dev, rank, world, with_e2e=(world == 1))
        door = run_door(dev, rank, world, (clocks or {}).get("sm_max_mhz"), props.multi_processor_count,
                        with_cpu=(world == 1 and not args.no_cpu_baseline))
        peg = run_door(dev, rank, world, (clocks or {}).get("sm_max_mhz"), props.multi_processor_count,
                       with_cpu=(world == 1 and not args.no_cpu_baseline), task="sawyer_peg")
        kit = run_kitchen(dev, rank, world, (clocks or {}).get("sm_max_mhz"), props.multi_processor_count,
                          with_cpu=(world == 1 and not args.no_cpu_baseline))

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        for pt in sweep:
            pt["frac"] = pt["achieved"] / peak
        achieved = ALG_BYTES_PER_ENV_STEP * n / per_launch_s / 1e9
        traffic, traffic_src = (args.traffic_bytes, "--traffic-bytes") if args.traffic_bytes is not None else ncu_traffic(n)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": per_launch_s * 1e3, "timed_region_s": ms * 1e-3,
                "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "state_dtype": "float32",
                "dtype_note": "arithmetic in fp64 (explicit round-to-nearest), state STORED as fp32 between steps (the 113-B layout): "
                              "one step from fp32-representable states is bit-exact; the sweep's float64 point keeps fp64 state "
                              "and is bit-exact over whole rollouts",
                "data": "synthetic", "config": config_dict(args, n_total),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * world,
                        "d2h_bytes_per_step": d2h * world, "steps": e2e_steps,
                        "api": "PersistentStateWrapper.step(pinned host actions) -> host obs/reward/done/success (earl_step_host: " + host_path_note() + ")",
                        "pcie_ceiling": ceiling,
                        "frac_of_pcie_ceiling": (e2e_value / ceiling["value"]) if ceiling else None},
                "gpu_launches": launches,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                             "kernel": ("earl::tabletop_step_kernel<false,true,1>  (persistent LSU kernel, PDL)" if n <= 3 * 1024 * 1024
                                        else "earl::tabletop_step_tile_kernel  (one 256-env tile per CTA, PDL)"),
                             "note": "per-env state (24 B) stays L2-resident at this batch size, so the algorithmic-byte "
                                     "rate can exceed the HBM copy peak; frac_all_hbm is the operating point where state, "
                                     "actions and outputs all stream from HBM (8,388,608 envs per GPU)",
                             "frac_all_hbm": (big["achieved"] / peak) if big else None,
                             "achieved_all_hbm": big["achieved"] if big else None,
                             "algorithmic_bytes_per_launch": ALG_BYTES_PER_ENV_STEP * n,
                             "avg_launch_us": per_launch_s * 1e6},
                "clocks": clocks}
        if big is not None:
            line["hbm_bound_check"] = big
        if sweep:
            line["sweep"] = sweep
        if collective is not None:
            line["eval_collective"] = collective
        if tt3 is not None:
            tt3["frac"] = tt3["achieved"] / peak
            line["tabletop_3obj"] = tt3
        if door is not None:
            line["sawyer_door"] = door
        if peg is not None:
            line["sawyer_peg"] = peg
        if kit is not None:
            line["kitchen"] = kit
        if world == 1 and not args.no_cpu_baseline and not args.profile:
            threads = os.cpu_count() or 1
            rate, n_sample, el, k = cpu_port_rate(n, min(args.steps, 200), threads, budget_s=15.0, min_wall_s=1.5)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"{n_sample} envs x {k} steps of the same workload, "
                                              f"step-major C oracle, OpenMP {threads} threads, {el:.2f} s ({el * threads:.0f} core-seconds)",
                                    "note": "a C restatement of the reference arithmetic, ~2e4 x faster per core than the reference's "
                                            "own Python loop (reference_python_loop: measured in the build container, where "
                                            "/root/reference exists, by oracle/ref_python_rate.py)",
                                    "reference_python_loop": ref_python_loop()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000, help="timed steps of the device-resident run (and of e2e by default)")
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--num-envs", type=int, default=1 << 20, help="envs per GPU")
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-hbm-check", action="store_true", help="skip the 8M-env all-HBM operating point")
    ap.add_argument("--no-door", action="store_true", help="skip the sawyer_door / sawyer_peg sections")
    ap.add_argument("--profile", action="store_true", help="under ncu: no sustained warm-up, 1 e2e step, no CPU leg")
    ap.add_argument("--traffic-bytes", type=float, default=None,
                    help="dram bytes per launch of the step kernel; default: looked up by batch size in "
                         "profiles/ncu_traffic.json (committed `ncu --set full` captures), else null")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the observations, rewards and dones of the last timed step (rank 0's "
                         "envs) as DIR/{obs,reward,done}.npy, float32; a seeded sample of envs beyond 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29577", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
