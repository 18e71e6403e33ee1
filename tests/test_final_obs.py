"""final_obs=True (EARL_FLAG_FINAL_OBS) without a GPU: the Python constructors and EARLEnvs reject it without auto_reset
before any library call, EARLEnvs hands it to the train env only, and every create entry point validates the flag before it
looks for a device."""
import ctypes
import functools
import os
import subprocess
import sys

import pytest

import earl_benchmark_b200 as eb
from conftest import REPO
from earl_benchmark_b200 import _lib
from earl_benchmark_b200.envs import kitchen, sawyer_door, sawyer_peg, tabletop_manipulation, tabletop_manipulation_3obj

CLASSES = {
    "tabletop_manipulation": tabletop_manipulation.TabletopManipulation,
    "tabletop_manipulation_3obj": tabletop_manipulation_3obj.TabletopManipulation,
    "sawyer_door": sawyer_door.SawyerDoorV2,
    "sawyer_peg": sawyer_peg.SawyerPegV2,
    "kitchen": kitchen.Kitchen,
}
LOADER = ["tabletop_manipulation", "sawyer_door", "sawyer_peg", "kitchen"]


@pytest.fixture
def no_library(monkeypatch):
    def refuse():
        raise AssertionError("the library was called")
    monkeypatch.setattr(_lib, "lib", refuse)


def reward(name):
    return "dense" if name == "kitchen" else "sparse"


@pytest.mark.parametrize("name", list(CLASSES))
def test_constructor_rejects_final_obs_without_auto_reset(name, no_library):
    with pytest.raises(ValueError, match="auto_reset"):
        CLASSES[name](reward_type=reward(name), num_envs=4, final_obs=True)


@pytest.mark.parametrize("name", list(CLASSES))
def test_constructor_accepts_final_obs_with_auto_reset(name):
    env = CLASSES[name](reward_type=reward(name), num_envs=4, auto_reset=True, final_obs=True)
    assert env._keep_final_obs and env._handle is None and env._final_obs is None   # lazy: nothing on a device yet


@pytest.mark.parametrize("name", list(CLASSES))
def test_flag_reaches_the_config_only_when_asked(name):
    env = CLASSES[name](reward_type=reward(name), num_envs=4, auto_reset=True)
    assert not env._keep_final_obs
    if name == "tabletop_manipulation":
        assert not env._flags() & _lib.FLAG_FINAL_OBS
        flagged = CLASSES[name](reward_type="sparse", num_envs=4, auto_reset=True, final_obs=True)
        assert flagged._flags() & _lib.FLAG_FINAL_OBS == _lib.FLAG_FINAL_OBS


@pytest.mark.parametrize("name", LOADER)
def test_loader_rejects_final_obs_without_auto_reset(name, no_library):
    with pytest.raises(ValueError, match="auto_reset"):
        eb.EARLEnvs(name, reward_type=reward(name), num_envs=4, final_obs=True)


@pytest.mark.parametrize("lifelong", [False, True])
@pytest.mark.parametrize("name", LOADER)
def test_loader_gives_final_obs_to_the_train_env_only(name, lifelong):
    envs = eb.EARLEnvs(name, reward_type=reward(name), num_envs=4, auto_reset=True, final_obs=True,
                       setup_as_lifelong_learning=lifelong).get_envs()
    train = envs if lifelong else envs[0]
    base = train
    while hasattr(base, "env"):
        base = base.env
    assert base._keep_final_obs and base._auto_reset
    if not lifelong:
        assert not envs[1].env._keep_final_obs and not envs[1].env._auto_reset
    plain = eb.EARLEnvs(name, reward_type=reward(name), num_envs=4, auto_reset=True).get_envs()[0]
    assert not plain.env._keep_final_obs


def without_gpu(test):
    """Run `test` where no GPU is visible: in this process on a machine without one, else in a child pytest that is shown
    none (CUDA_VISIBLE_DEVICES empty), so the create-time checks are seen to come before any device is looked for."""
    @functools.wraps(test)
    def run():
        import torch
        if not torch.cuda.is_available():
            return test()
        r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", f"{os.path.abspath(__file__)}::{test.__name__}"],
                           cwd=REPO, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    return run


def create_codes(flags):
    """earl_*_create return codes and messages of the four tasks for `flags` (no handle can come out without a device)"""
    L = _lib.lib()
    out = {}
    h = ctypes.c_void_p()
    cfg = _lib.EarlConfig(_lib.ENV_TABLETOP, 4, 0, flags, 10, 0, 1, 0)
    blob = tabletop_manipulation.TabletopManipulation(num_envs=4, device="cuda:0")._model_blob()
    out["tabletop"] = L.earl_create(ctypes.byref(cfg), ctypes.byref(blob), ctypes.sizeof(blob), ctypes.byref(h)), L.earl_last_error()
    t3 = _lib.Tt3Config()
    t3.num_envs, t3.num_goals, t3.episode_horizon, t3.flags = 4, 1, 10, flags
    out["tt3"] = L.earl_tt3_create(ctypes.byref(t3), ctypes.sizeof(t3), ctypes.byref(h)), L.earl_last_error()
    door = sawyer_door.SawyerDoorV2(num_envs=4, device="cuda:0")
    mj = _lib.MjConfig(_lib.ENV_SAWYER_DOOR, 4, 0, flags, 10, 0)
    blob = door.model.to_blob()
    task = door._task_spec()
    out["door"] = L.earl_mj_create(ctypes.byref(mj), blob, len(blob), ctypes.byref(task), ctypes.byref(h)), L.earl_last_error()
    k = kitchen.MjkConfig()
    k.num_envs, k.frame_skip, k.episode_horizon, k.flags = 4, 40, 10, flags
    kb = kitchen.Kitchen(num_envs=4, device="cuda:0").model.to_blob()
    out["kitchen"] = L.earl_mjk_create(ctypes.byref(k), kb, len(kb), ctypes.byref(h)), L.earl_last_error()
    return out


@without_gpu
def test_create_validates_the_flag_before_looking_for_a_device():
    import torch
    assert not torch.cuda.is_available()
    for task, (rc, msg) in create_codes(_lib.FLAG_FINAL_OBS).items():
        assert rc == -1 and b"EARL_FLAG_FINAL_OBS needs EARL_FLAG_AUTO_RESET" in msg, (task, rc, msg)
    for task, (rc, msg) in create_codes(_lib.FLAG_FINAL_OBS | _lib.FLAG_AUTO_RESET).items():
        assert rc != 0 and b"FINAL_OBS" not in msg, (task, rc, msg)        # accepted: it fails later, for want of a device
    L = _lib.lib()
    for fn in ("earl_set_final_obs", "earl_tt3_set_final_obs", "earl_mj_set_final_obs", "earl_mjk_set_final_obs"):
        assert getattr(L, fn)(None, None) == -1, fn
