"""Kitchen evaluation statistics without a device: the loader asks for them on the eval env only, and a statistics handle
fails loudly where there is no GPU (no CPU path)."""
import functools
import os
import subprocess
import sys

import pytest

from conftest import REPO
from earl_benchmark_b200 import _lib


def without_gpu(test):
    """Run `test` where no GPU is visible: in this process on a machine without one, else in a child pytest that is shown
    none (CUDA_VISIBLE_DEVICES empty)."""
    @functools.wraps(test)
    def run():
        import torch
        if not torch.cuda.is_available():
            return test()
        r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", f"{os.path.abspath(__file__)}::{test.__name__}"],
                           cwd=REPO, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    return run


def test_loader_configures_statistics_on_the_kitchen_eval_env_only():
    import earl_benchmark_b200 as eb
    tr, ev = eb.EARLEnvs("kitchen", reward_type="dense", num_envs=4).get_envs()   # lazy: no device needed
    assert ev.env._eval_stats is True and tr.env._eval_stats is False
    _, ev = eb.EARLEnvs("kitchen", reward_type="dense", num_envs=4, eval_stats=False).get_envs()
    assert ev.env._eval_stats is False
    tr = eb.EARLEnvs("kitchen", reward_type="dense", setup_as_lifelong_learning=True, num_envs=4).get_envs()
    assert tr.env._eval_stats is False


@without_gpu
def test_kitchen_statistics_handle_has_no_cpu_fallback():
    import torch
    assert not torch.cuda.is_available()
    from earl_benchmark_b200.envs import kitchen
    env = kitchen.Kitchen(num_envs=2, eval_stats=True)                # construction is lazy: host constants only
    assert env._eval_stats is True
    with pytest.raises(_lib.EarlError) as ei:
        env.reset()
    assert ei.value.code == -2                                        # EARL_ERR_CUDA, not a rejected flag
