"""Multi-GPU plumbing: one process per GPU, environments sharded by index, NO collective on the step path.

The only collective of the system is one small all-reduce of per-evaluation statistics
(sum of returns, success counts, env count) -- NCCL over NVLink/NVSwitch on GPUs, gloo in CPU tests.
The reference has no counterpart (it is single-process, SURVEY.md section 2.2).
"""
import os

import torch
import torch.distributed as dist


def init_from_env(backend=None):
    """Initialise torch.distributed from torchrun's environment (no-op for single-process runs).
    Returns (rank, world_size, local_rank)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
        dist.init_process_group(backend=backend, rank=rank, world_size=world,
                                device_id=torch.device("cuda", local) if backend == "nccl" else None)
    return rank, world, local


def all_reduce_eval_stats(stats, group=None):
    """Sum the [4] float64 statistics tensor of an env's `eval_stats()` over all ranks, in place: the tabletop, the
    three-object tabletop, sawyer_door, sawyer_peg and kitchen envs built with `eval_stats=True`.

    stats = (sum of episode returns, #envs successful at their last step, #envs successful at any step, N).
    Returns a dict with the job-wide means."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    s = stats.detach().cpu().tolist()
    n = max(s[3], 1.0)
    return {"mean_return": s[0] / n, "success_rate": s[1] / n, "success_any_rate": s[2] / n, "num_envs": int(s[3])}


def max_over_ranks(value, device=None):
    """Max of a Python float over ranks (timing: a multi-GPU step takes as long as its slowest rank)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())
