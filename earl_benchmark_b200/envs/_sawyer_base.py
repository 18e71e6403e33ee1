"""Shared machinery of the batched Sawyer envs (door, peg): handle lifetime, stepping (device and host paths), goal
table, counters, statistics and state access over the C ABI of include/earl_mj_b200.h.  Task classes
(envs/sawyer_door.py, envs/sawyer_peg.py) supply the model file, the task constants and the reset draws.
Without the CUDA library or a CUDA device everything here raises; there is no CPU path."""
import ctypes as C
import os

import numpy as np
import torch

from .. import _lib, rng
from ._goals import goal_args
from ._hostio import HostBuffers
from ..mjcf.compile import Model
from ..spaces import Box

OBS_DIM, ACT_DIM = 14, 4
_NEVER = 1 << 62
MODEL_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "models")


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


class SawyerBatchedEnv:
    """N independent Sawyer envs stepped by one kernel launch (one warp per env)."""
    ENV_KIND = None          # _lib.ENV_SAWYER_*
    MODEL_FILE = None        # file under models/
    SUCCESS_RADIUS = None
    HAS_DENSE_REWARD = False

    def __init__(self, reward_type="sparse", reset_at_goal=False, num_envs=1, device=None, seed=0, eval_stats=False,
                 env_offset=0, total_envs=None, model_path=None, max_newton=0, host_io=False, auto_reset=False,
                 reset_stream_rows=64, per_env_goals=False, final_obs=False, **_tabletop_only):
        name = type(self).__name__
        if final_obs and not auto_reset:
            raise ValueError("final_obs=True needs auto_reset=True: without it, the observation step() returns on done is the final one")
        if reward_type == "dense" and not self.HAS_DENSE_REWARD:
            raise NotImplementedError(f"{name}: the dense reward (metaworld reward_utils, gripper caging) is not built yet")
        if reward_type not in ("sparse", "dense"):
            raise ValueError(f"reward_type must be 'sparse' or 'dense', got {reward_type!r}")
        self._reward_type = reward_type
        self._reset_at_goal = bool(reset_at_goal)
        self.num_envs = int(num_envs)
        self._seed = int(seed)
        self._eval_stats = bool(eval_stats)
        self._env_offset = int(env_offset)
        self._total_envs = int(total_envs) if total_envs is not None else self.num_envs + self._env_offset
        self._max_newton = int(max_newton)
        if device is None:
            device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        self.device = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        if self.device.type != "cuda":
            raise ValueError("earl_benchmark_b200 environments live on a CUDA device; there is no CPU path")
        self.model = Model.load(model_path or os.path.join(MODEL_DIR, self.MODEL_FILE))
        self.max_path_length = int(1e8)
        self.action_space = Box(-1.0, 1.0, (ACT_DIM,), np.float32)
        self.observation_space = Box(-np.inf, np.inf, (OBS_DIM,), np.float32)
        self._goal_table = []
        self._episode_horizon = _NEVER
        self._lifelong = False
        self._goal_change_frequency = 0
        self._handle = None
        self._np_random = rng.NumpyLegacyRandom(self._seed & 0xFFFFFFFF)
        self._obs = self._reward = self._done = self._success = self._final_obs = None
        self._host_bufs = None
        self._host_mode = bool(host_io)   # host_io=True: reset() returns numpy like the numpy-driven step()
        # auto_reset=True: an env whose horizon fires is reset inside step() on the device, and every reset without an
        # override takes its draws from a pre-drawn stream of `reset_stream_rows` full resets per env (see reset_stream())
        self._auto_reset = bool(auto_reset)
        self._reset_stream_rows = int(reset_stream_rows)
        if self._reset_stream_rows < 1:
            raise ValueError("reset_stream_rows must be >= 1")
        # per_env_goals=True: every env can be given its own goal vector, effective at once (set_goals / get_goals)
        self._per_env_goals = bool(per_env_goals)
        # final_obs=True (with auto_reset): every step's info["final_observation"] holds the last observation of each
        # episode the step ended (see step())
        self._keep_final_obs = bool(final_obs)

    # ------------------------------------------------------------------ task hooks
    def _task_spec(self):
        raise NotImplementedError

    def _draw_reset(self, mask):
        """-> (obj_qpos float64 [N,k], goal rows int32 [N] or None): the random draws of reset_model(), env order."""
        raise NotImplementedError

    def _reset_stream(self, rows):
        """-> (obj_qpos float64 [rows,N,k], goal rows int32 [rows,N] or None): this shard's columns of the pre-drawn
        reset stream of an auto-reset handle."""
        raise NotImplementedError

    # ------------------------------------------------------------------ construction
    def _configure(self, episode_horizon=None, lifelong=None, goal_change_frequency=None):
        if self._handle is not None:
            raise RuntimeError("wrappers must be applied before the env is first reset/stepped")
        if episode_horizon is not None:
            self._episode_horizon = int(episode_horizon)
        if lifelong is not None:
            if lifelong and self._reset_at_goal and type(self).__name__ == "SawyerPegV2":
                raise NotImplementedError("SawyerPegV2: lifelong goal swaps with reset_at_goal (random goals) are not built")
            self._lifelong = bool(lifelong)
        if goal_change_frequency is not None:
            self._goal_change_frequency = int(goal_change_frequency)

    def _ensure(self):
        if self._handle is not None:
            return
        L = _lib.lib()
        flags = (_lib.FLAG_EVAL_STATS if self._eval_stats else 0) | (_lib.FLAG_LIFELONG if self._lifelong else 0)
        flags |= _lib.FLAG_AUTO_RESET if self._auto_reset else 0
        flags |= _lib.FLAG_PER_ENV_GOALS if self._per_env_goals else 0
        flags |= _lib.FLAG_FINAL_OBS if self._keep_final_obs else 0
        if self._reward_type == "dense":
            flags |= _lib.FLAG_DENSE_REWARD
        cfg = _lib.MjConfig(self.ENV_KIND, self.num_envs, self.device.index or 0, flags, self._episode_horizon,
                            self._goal_change_frequency)
        blob = self.model.to_blob()
        task = self._task_spec()
        h = C.c_void_p()
        _lib.check(L.earl_mj_create(C.byref(cfg), blob, len(blob), C.byref(task), C.byref(h)))
        self._handle = h
        self._upload_goals()
        # sim.reset() + _reset_hand(50) with ctrl [-1, 1] (SawyerXYZEnv._reset_hand), simulated once on the device
        hand = np.ascontiguousarray(np.asarray(self.hand_init_pos, np.float64))
        ctrl = np.array([-1.0, 1.0], np.float32)
        _lib.check(L.earl_mj_build_reset_template(h, hand.ctypes.data, ctrl.ctypes.data, 50))
        n, dev = self.num_envs, self.device
        self._obs = torch.empty((n, OBS_DIM), dtype=torch.float32, device=dev)
        self._reward = torch.empty((n,), dtype=torch.float32, device=dev)
        self._done = torch.empty((n,), dtype=torch.uint8, device=dev)
        self._success = torch.empty((n,), dtype=torch.uint8, device=dev)
        self._goal_rows = torch.zeros((n,), dtype=torch.int32, device=dev)   # the handle reads it (auto reset): never rebound
        if self._keep_final_obs:   # rows of envs that have not ended an episode yet hold NaN
            self._final_obs = torch.full((n, OBS_DIM), float("nan"), dtype=torch.float32, device=dev)
            _lib.check(L.earl_mj_set_final_obs(h, self._final_obs.data_ptr()))
        if self._auto_reset:
            qpos, rows = self._reset_stream(self._reset_stream_rows)
            qpos = np.ascontiguousarray(qpos, np.float64)
            rows = None if rows is None else np.ascontiguousarray(rows, np.int32)
            _lib.check(L.earl_mj_set_reset_stream(h, qpos.ctypes.data, None if rows is None else rows.ctypes.data,
                                                  self._reset_stream_rows, self._goal_rows.data_ptr()))

    def _upload_goals(self):
        g = np.ascontiguousarray(np.stack(self._goal_table), np.float64)
        _lib.check(_lib.lib().earl_mj_set_goal_table(self._handle, g.ctypes.data, len(g)))

    def close(self):
        if self._handle is not None:
            _lib.lib().earl_mj_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ goals
    def _goal_row(self, g):
        g = np.asarray(g, np.float64).reshape(7)
        for r, t in enumerate(self._goal_table):
            if np.array_equal(t, g):
                return r
        self._goal_table.append(g.copy())
        if self._handle is not None:
            self._upload_goals()
        return len(self._goal_table) - 1

    def reset_goal(self, goal=None):
        """goal: None (the task's next goal) or one 7-vector shared by all envs.  Takes effect at the next reset."""
        self._ensure()
        if goal is None:
            goal = self.get_next_goal()[0]
        self._goal_rows.fill_(self._goal_row(goal))

    @property
    def goal(self):
        return np.stack([self._goal_table[r] for r in self._goal_rows.cpu().numpy()])

    def set_goals(self, goals, mask=None):
        """reset_goal(goal) with any goal per env, effective at once (per_env_goals=True envs only).

        goals: CUDA float32 / float64 tensor [N,7], or [7] for every env; mask: CUDA bool / uint8 [N] or None (all envs).
        The masked envs pursue their new goal from now on: the returned observation [N,14] carries it (the other rows are
        the current observation) and the next step's reward (sparse and dense), success, statistics and lifelong return are
        measured against it.  float64 goals are rounded to float32 as the goal table rounds them.  The goal the next reset
        assigns (reset_goal) is unchanged, so a reset, auto-reset or lifelong goal swap gives the env the task's goal back.
        One launch on the current stream, no synchronisation.  host_io=True envs also take numpy / CPU input and return
        numpy."""
        if not self._per_env_goals:
            raise RuntimeError("set_goals needs an env built with per_env_goals=True")
        self._ensure()
        g, dtype, m = goal_args(goals, mask, self.num_envs, 7, self.device, self._host_mode)
        obs = torch.empty((self.num_envs, OBS_DIM), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().earl_mj_set_goals(self._handle, g.data_ptr(), dtype, _ptr(m), obs.data_ptr(), _stream()))
        return obs.cpu().numpy() if self._host_mode else obs

    def get_goals(self):
        """CUDA float32 [N,7]: the goal every env pursues now (per_env_goals=True envs only)."""
        if not self._per_env_goals:
            raise RuntimeError("get_goals needs an env built with per_env_goals=True")
        self._ensure()
        out = torch.empty((self.num_envs, 7), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().earl_mj_get_goals(self._handle, out.data_ptr(), _stream()))
        return out

    # ------------------------------------------------------------------ reset / step
    def _mask(self, mask):
        if mask is None:
            return None
        return torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()

    def _reset_device(self, m, obj_qpos):
        """obj_qpos None (auto-reset handles): each reset env's next draw of the pre-drawn reset stream."""
        a = None if obj_qpos is None else torch.as_tensor(np.array(obj_qpos, np.float64, order="C", copy=True)).to(self.device)
        obs = torch.empty((self.num_envs, OBS_DIM), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().earl_mj_reset(self._handle, _ptr(m), _ptr(a), self._goal_rows.data_ptr(), obs.data_ptr(), _stream()))
        if m is not None:  # rows of envs that were not reset still need their current observation
            obs = torch.where(m.view(-1, 1).bool(), obs, self._get_obs())
        return obs.cpu().numpy() if self._host_mode else obs   # numpy-driven env: numpy out, like its step()

    def step(self, action, out=None):
        """One step of every env.  CUDA float32 tensor [N,4] -> CUDA tensors (obs [N,14], reward [N], done [N] bool,
        info), owned by the env and valid until the next step; numpy / CPU tensor -> host path, numpy arrays.
        final_obs=True envs add info["final_observation"] [N,14]: on rows where done is set, the observation the step
        reached before the auto-reset replaced it; other rows keep what an earlier step stored there (NaN before an env's
        first episode ends).  The env-owned tensor, valid until the next step; a numpy copy on the host path."""
        self._ensure()
        if isinstance(action, torch.Tensor) and action.is_cuda:
            a = action
            if a.dtype != torch.float32 or not a.is_contiguous():
                a = a.to(torch.float32).contiguous()
            if a.numel() != self.num_envs * ACT_DIM:
                raise ValueError(f"action must have shape [{self.num_envs},{ACT_DIM}]")
            obs, rew, done, succ = out if out is not None else (self._obs, self._reward, self._done, self._success)
            _lib.check(_lib.lib().earl_mj_step(self._handle, a.data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr(),
                                               _ptr(succ), _stream()))
            info = {"success": None if succ is None else succ.view(torch.bool)}
            if self._final_obs is not None:
                info["final_observation"] = self._final_obs
            return obs, rew, done.view(torch.bool), info
        return self._step_host(action)

    def _step_host(self, action):
        """numpy / CPU-tensor step: H2D copy, kernel, D2H copies inside one C call; returns numpy arrays that stay valid
        until the step after next (two alternating pinned output sets, envs/_hostio.py)."""
        if self._host_bufs is None:
            self._host_bufs = HostBuffers(self.num_envs, ACT_DIM, OBS_DIM)
        hb = self._host_bufs
        src = hb.stage(action)
        ho, hr, hd, hs = hb.next_outputs()
        _lib.check(_lib.lib().earl_mj_step_host(self._handle, src.data_ptr(), ho.data_ptr(), hr.data_ptr(), hd.data_ptr(),
                   hs.data_ptr()))
        return HostBuffers.as_numpy(ho, hr, hd, hs, self._final_obs)

    def _get_obs(self):
        self._ensure()
        obs = torch.empty((self.num_envs, OBS_DIM), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().earl_mj_get_obs(self._handle, obs.data_ptr(), _stream()))
        return obs

    def get_obs(self):
        return self._get_obs()

    def is_successful(self, obs=None):
        """||obs[4:7] - obs[11:14]|| <= radius (sawyer_door.py:173-177, sawyer_peg.py:301-305) on caller-supplied
        observations (cold path; the step kernel computes the same test for the states it produces)."""
        if obs is None:
            obs = self._get_obs()
        if isinstance(obs, torch.Tensor):
            o = obs.reshape(-1, OBS_DIM)
            return torch.linalg.norm(o[:, 4:7] - o[:, 11:14], dim=1) <= self.SUCCESS_RADIUS
        o = np.asarray(obs).reshape(-1, OBS_DIM)
        return np.linalg.norm(o[:, 4:7] - o[:, 11:14], axis=1) <= self.SUCCESS_RADIUS

    def compute_reward(self, obs, actions=None):
        """Sparse reward of caller-supplied observations (cold path; task classes with a dense reward override this)."""
        s = self.is_successful(obs)
        return s.to(torch.float32) if isinstance(s, torch.Tensor) else s.astype(np.float32)

    # ------------------------------------------------------------------ counters / stats / state
    def _counters(self, want_ll=False):
        self._ensure()
        total = C.c_int64()
        n = self.num_envs
        interv = torch.empty((n,), dtype=torch.int64, device=self.device)
        since = torch.empty((n,), dtype=torch.int32, device=self.device)
        ll = torch.empty((n,), dtype=torch.float64, device=self.device) if want_ll else None
        _lib.check(_lib.lib().earl_mj_counters(self._handle, C.byref(total), interv.data_ptr(), since.data_ptr(), _ptr(ll), _stream()))
        return total.value, interv, since, ll

    def eval_stats(self):
        self._ensure()
        out = torch.empty((4,), dtype=torch.float64, device=self.device)
        _lib.check(_lib.lib().earl_mj_eval_stats(self._handle, out.data_ptr(), _stream()))
        return out

    def work_counters(self):
        """dict of work done by the step kernel since creation (env_steps, substeps, newton_iterations, ...)."""
        self._ensure()
        out = np.zeros(7, np.uint64)
        _lib.check(_lib.lib().earl_mj_work_counters(self._handle, out.ctypes.data))
        d = dict(zip(("env_steps", "substeps", "newton_iterations", "constraint_rows", "contacts", "bad_states",
                      "overflow_states"),
                     (int(x) for x in out)))
        d["redone_states"] = int(_lib.lib().earl_mj_redo_count(self._handle))   # re-stepped by the extra-large capacity set
        return d

    @property
    def launch_count(self):
        return 0 if self._handle is None else int(_lib.lib().earl_mj_launch_count(self._handle))

    def get_state(self):
        """Physics state as host arrays: dict(qpos [N,nq], qvel [N,nv], qacc_warmstart [N,nv], mocap_pos [N,3])."""
        self._ensure()
        n, nq, nv = self.num_envs, int(self.model.nq), int(self.model.nv)
        q, v, w, mp = np.zeros((n, nq)), np.zeros((n, nv)), np.zeros((n, nv)), np.zeros((n, 3))
        _lib.check(_lib.lib().earl_mj_get_state(self._handle, q.ctypes.data, v.ctypes.data, w.ctypes.data, mp.ctypes.data))
        return dict(qpos=q, qvel=v, qacc_warmstart=w, mocap_pos=mp)

    def set_state(self, qpos=None, qvel=None, qacc_warmstart=None, mocap_pos=None):
        self._ensure()
        n = self.num_envs

        def arr(a, w):
            if a is None:
                return None, 0
            x = np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), (n, w)))
            return x, x.ctypes.data
        nq, nv = int(self.model.nq), int(self.model.nv)
        keep = [arr(qpos, nq), arr(qvel, nv), arr(qacc_warmstart, nv), arr(mocap_pos, 3)]
        _lib.check(_lib.lib().earl_mj_set_state(self._handle, *[k[1] for k in keep]))
