"""Argument checks of `set_goals()` (per-env goals, `per_env_goals=True`), shared by the tabletop and Sawyer env classes.

Everything here reads tensor metadata only: no value of the goals or the mask is looked at on the host, so `set_goals()`
stays one launch on the current stream with no synchronisation."""
import numpy as np
import torch

from .. import _lib


def goal_args(goals, mask, num_envs, width, device, host_io):
    """-> (goals [num_envs, width] contiguous CUDA float32/float64 tensor, EARL_GOAL_* code, mask uint8 [num_envs] or None).

    goals: [num_envs, width] or [width] (the same goal for every env); mask: [num_envs] bool / uint8 or None.  A CUDA
    tensor is required unless the env was built with host_io=True, which also takes numpy arrays and CPU tensors."""
    index = device.index if device.index is not None else torch.cuda.current_device()

    def on_device(x, what):
        if isinstance(x, torch.Tensor) and x.is_cuda:
            if x.device.index != index:
                raise ValueError(f"{what} is on {x.device}, the env on {device}")
            return x
        if not host_io:
            raise TypeError(f"{what} must be a CUDA tensor (numpy / CPU input is taken by host_io=True envs only)")
        return torch.as_tensor(np.asarray(x) if not isinstance(x, torch.Tensor) else x).to(device)

    g = on_device(goals, "goals")
    if g.dtype not in (torch.float32, torch.float64):
        raise TypeError(f"goals must be float32 or float64, got {g.dtype}")
    if g.dim() == 1 and g.shape[0] == width:
        g = g.expand(num_envs, width)
    elif g.dim() != 2 or tuple(g.shape) != (num_envs, width):
        raise ValueError(f"goals must have shape [{num_envs},{width}] or [{width}], got {list(g.shape)}")
    g = g.contiguous()
    m = None
    if mask is not None:
        m = on_device(mask, "mask")
        if m.dtype not in (torch.bool, torch.uint8):
            raise TypeError(f"mask must be bool or uint8, got {m.dtype}")
        if tuple(m.shape) != (num_envs,):
            raise ValueError(f"mask must have shape [{num_envs}], got {list(m.shape)}")
        m = m.contiguous().view(torch.uint8)
    return g, (_lib.GOAL_F64 if g.dtype == torch.float64 else _lib.GOAL_F32), m
