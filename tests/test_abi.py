"""The C-ABI library loads on a CPU-only box and exports every symbol include/earl_b200.h declares."""
import ctypes
import functools
import os
import re
import subprocess
import sys

import pytest

from conftest import REPO
from earl_benchmark_b200 import _lib, build

HEADERS = [os.path.join(REPO, "include", f) for f in ("earl_b200.h", "earl_tt3_b200.h", "earl_mj_b200.h", "earl_mj_kitchen_b200.h")]


def header_symbols():
    text = "\n".join(open(h).read() for h in HEADERS)
    return re.findall(r"^EARL_API\s+[\w\s\*]+?\b(earl_\w+)\s*\(", text, flags=re.M)


def test_library_builds_and_loads():
    build.build()
    L = _lib.lib()
    assert L.earl_abi_version() == _lib.EARL_ABI_VERSION


def test_every_declared_symbol_is_exported_and_bound():
    build.build()
    syms = header_symbols()
    assert len(syms) >= 25 and len(set(syms)) == len(syms)
    L = ctypes.CDLL(_lib.LIB_PATH)
    for s in syms:
        assert hasattr(L, s), f"{s} declared in the header but not exported"
    bound = {name for name, _, _ in _lib.SIGNATURES}
    assert bound == set(syms), (bound ^ set(syms))
    exported = subprocess.check_output(["nm", "-D", "--defined-only", _lib.LIB_PATH], text=True)
    extra = [l.split()[-1] for l in exported.splitlines() if " T " in l and not l.split()[-1].startswith("earl_")]
    assert not extra, f"non-API symbols exported: {extra}"


def test_struct_layouts_match_header():
    # sizes the C side checks against (earl_create rejects blobs of any other size)
    assert ctypes.sizeof(_lib.EarlConfig) == 40
    assert ctypes.sizeof(_lib.TabletopModel) == 8 + 4 * 8 + 6 * 8 + 256 * 6 * 8
    assert ctypes.sizeof(_lib.MjConfig) == 32
    assert ctypes.sizeof(_lib.Tt3Config) == 16 + 8 + 4 * 8 + 10 * 8 + 16 * 10 * 8
    assert ctypes.sizeof(_lib.MjTask) == 8 * 4 + 8 * 4 + 6 * 4 + 7 * 4


def without_gpu(test):
    """Run `test` where no GPU is visible: in this process on a machine without one, else in a child pytest that is shown
    none (CUDA_VISIBLE_DEVICES empty), so the no-fallback checks run on GPU machines too."""
    @functools.wraps(test)
    def run():
        import torch
        if not torch.cuda.is_available():
            return test()
        r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", f"{os.path.abspath(__file__)}::{test.__name__}"],
                           cwd=REPO, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    return run


@without_gpu
def test_no_cpu_fallback_without_gpu():
    import torch
    assert not torch.cuda.is_available()
    import earl_benchmark_b200 as e
    tr, _ = e.EARLEnvs("tabletop_manipulation", num_envs=4).get_envs()
    with pytest.raises(_lib.EarlError) as ei:
        tr.reset()
    assert ei.value.code == -2  # EARL_ERR_CUDA: fails loudly, no silent CPU path


@without_gpu
def test_kitchen_has_no_cpu_fallback_either():
    import torch
    assert not torch.cuda.is_available()
    import numpy as np
    from earl_benchmark_b200.envs import kitchen
    env = kitchen.Kitchen(num_envs=2)           # construction is lazy: host constants only
    assert env.get_init_states().shape == (6, 23)
    with pytest.raises(_lib.EarlError) as ei:
        env.reset()
    assert ei.value.code == -2                  # EARL_ERR_CUDA
    from earl_benchmark_b200.kitchen_engine import KitchenEngine
    with pytest.raises(_lib.EarlError):
        KitchenEngine("cuda:0")
    assert np.array_equal(env.get_next_goal(), kitchen.goal_states[0])


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(REPO, "earl_benchmark_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".hpp", ".h")):
                text = open(os.path.join(root, f)).read()
                assert "oracle" not in text.replace("oracle/gen_golden.py", "").replace("tests/golden", ""), os.path.join(root, f)


def test_sqrt_free_thresholds_are_exact():
    """The kernels test s < attach_sq and s <= success_sq instead of taking square roots; both forms must
    agree with the reference's sqrt-then-compare for EVERY s, checked here around the boundary."""
    import numpy as np
    a, s = ctypes.c_double(), ctypes.c_float()
    _lib.lib().earl_tabletop_thresholds(0.4, 0.2, ctypes.byref(a), ctypes.byref(s))
    x = np.float64(a.value)
    xs = [x]
    lo = hi = x
    for _ in range(2000):
        lo, hi = np.nextafter(lo, 0.0), np.nextafter(hi, np.inf)
        xs += [lo, hi]
    xs = np.array(xs + list(np.random.RandomState(0).uniform(0, 1, 20000)))
    assert np.array_equal(np.sqrt(xs) < 0.4, xs < x)
    y = np.float32(s.value)
    ys = [y]
    lo = hi = y
    for _ in range(2000):
        lo, hi = np.nextafter(lo, np.float32(0)), np.nextafter(hi, np.float32(np.inf))
        ys += [lo, hi]
    ys = np.array(ys + list(np.random.RandomState(1).uniform(0, 0.2, 20000).astype(np.float32)), dtype=np.float32)
    assert np.array_equal(np.sqrt(ys).astype(np.float64) <= 0.2, ys <= y)


@without_gpu
def test_three_object_tabletop_has_no_cpu_fallback_and_validates_its_config():
    import torch
    L = _lib.lib()
    cfg = _lib.Tt3Config()
    h = ctypes.c_void_p()
    cfg.num_envs, cfg.num_goals, cfg.episode_horizon = 4, 1, 10
    assert L.earl_tt3_create(ctypes.byref(cfg), ctypes.sizeof(cfg) - 8, ctypes.byref(h)) == -1      # size check
    cfg.num_goals = 17
    assert L.earl_tt3_create(ctypes.byref(cfg), ctypes.sizeof(cfg), ctypes.byref(h)) == -1          # goal rows
    cfg.num_goals, cfg.flags = 1, _lib.FLAG_LIFELONG
    assert L.earl_tt3_create(ctypes.byref(cfg), ctypes.sizeof(cfg), ctypes.byref(h)) == -4          # unsupported flag
    assert b"three-object" in L.earl_last_error()
    assert not torch.cuda.is_available()
    from earl_benchmark_b200.envs.tabletop_manipulation_3obj import TabletopManipulation
    from earl_benchmark_b200.wrappers.persistent_state_wrapper import PersistentStateWrapper
    env = PersistentStateWrapper(TabletopManipulation(reward_type="sparse", num_envs=4), 100)
    assert env.get_next_goal().shape == (4, 10)         # host constants work without a device
    with pytest.raises(_lib.EarlError) as ei:
        env.reset()
    assert ei.value.code == -2                          # EARL_ERR_CUDA: fails loudly
