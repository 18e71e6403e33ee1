"""Pinned host buffers of the numpy / CPU-tensor step path (`earl_*_step_host`), shared by the env classes.

The reference returns FRESH arrays from every `step()`, so the canonical loop

    next_obs, r, done, _ = env.step(a); buffer.add(obs, a, r, next_obs); obs = next_obs

may hold `obs` across the next call.  Returning views of ONE pinned output set would make `obs` and `next_obs` the same
memory from the second step on (ADVICE r1).  Copying 56 MB per step at 1M envs would cost more than the PCIe transfer
it follows, so the outputs alternate between TWO pinned sets instead: the arrays a step returns stay untouched during
the NEXT step and are overwritten by the one after it ("valid until the step after next").  Anything kept longer must be
copied by the caller, as a replay buffer's `add` does.
"""
import numpy as np
import torch


class HostBuffers:
    def __init__(self, n, act_dim, obs_dim):
        pin = dict(pin_memory=True)
        self.n, self.act_dim, self.obs_dim = n, act_dim, obs_dim
        self.act = torch.empty((n, act_dim), dtype=torch.float32, **pin)
        self.sets = [(torch.empty((n, obs_dim), dtype=torch.float32, **pin), torch.empty((n,), dtype=torch.float32, **pin),
                      torch.empty((n,), dtype=torch.uint8, **pin), torch.empty((n,), dtype=torch.uint8, **pin)) for _ in range(2)]
        self.turn = 0

    def stage(self, action):
        """Pinned float32 [n, act_dim] tensor holding `action` (the caller's own tensor when it already is one)."""
        if isinstance(action, torch.Tensor):
            if action.is_pinned() and action.dtype == torch.float32 and action.is_contiguous() and action.numel() == self.n * self.act_dim:
                return action
            self.act.copy_(action.reshape(self.n, self.act_dim))
        else:
            self.act.numpy()[...] = np.asarray(action, np.float32).reshape(self.n, self.act_dim)
        return self.act

    def next_outputs(self):
        self.turn ^= 1
        return self.sets[self.turn]

    @staticmethod
    def as_numpy(ho, hr, hd, hs, final_obs=None):
        """numpy views of one output set; `final_obs` (the env's device buffer of final observations, final_obs=True envs)
        is added to info as a host copy, taken after the synchronous host step has written it"""
        info = {"success": hs.numpy().view(np.bool_)}
        if final_obs is not None:
            info["final_observation"] = final_obs.cpu().numpy()
        return ho.numpy(), hr.numpy(), hd.numpy().view(np.bool_), info


def ranks_on_this_host():
    """How many processes of this job drive a GPU from this host (torchrun's LOCAL_WORLD_SIZE / WORLD_SIZE, or the initialised
    process group): they share the host's PCIe root complex and memory bandwidth."""
    import os
    for key in ("LOCAL_WORLD_SIZE", "WORLD_SIZE"):
        v = os.environ.get(key)
        if v and v.isdigit():
            return max(1, int(v))
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_world_size()
    except Exception:
        pass
    return 1


def host_zerocopy_default():
    """Policy behind earl_set_host_zerocopy (include/earl_b200.h): None = EARL_TT_HOST_ZEROCOPY decides (read by the library),
    else 1 when this process has the host to itself and 0 when several ranks share it (measured: DESIGN.md section 4)."""
    import os
    if os.environ.get("EARL_TT_HOST_ZEROCOPY") is not None:
        return None
    return 1 if ranks_on_this_host() == 1 else 0

