"""Batched, device-resident three-object `TabletopManipulation`.

Mirror of the reference class `earl_benchmark/envs/tabletop_manipulation_3obj.py:20-165` (same constructor
arguments, method names and semantics: three draggable objects, the closest one within the threshold is
grasped) with a leading environment dimension on every array.  All arithmetic runs in the CUDA library
(csrc/earl_tt3.cu) through the C ABI of include/earl_tt3_b200.h; this file owns buffers and argument
marshalling.  Without the CUDA library or a CUDA device it raises.  Like the reference module it is not wired
into `EARLEnvs` (the reference's loader never constructs it either); wrap it in `PersistentStateWrapper`.

Differences a caller can observe:
  * every array has a leading [N] dimension; rewards / dones are arrays;
  * gym's constructor-time random `step()` is not replayed: call reset() first;
  * goals are rows of a goal table (`goal_states`; custom goals are appended, up to 16 rows);
  * `reset_at_goal` noise comes from a per-env-object replica of the legacy `np.random.seed(seed)` stream,
    consumed in env order (env 0's eight uniforms, then env 1's, ...), as a Python loop over N reference envs
    sharing the global stream would.  A full reset draws the eight uniforms of all `total_envs` envs of the job and
    keeps this shard's; a masked reset draws eight per selected env, in env order;
  * `auto_reset=True`: an env whose horizon fires is reset inside step(), on the device, with the same result as
    reset(mask=done).  With `reset_at_goal` too, every reset without `init_qpos` (auto or host) takes its qpos from a
    pre-drawn stream of `reset_stream_rows` rows per env (see reset_stream()), so the draws do not depend on when an
    env resets or on how the job is sharded.
"""
import ctypes as C

import numpy as np
import torch

from .. import _lib, rng
from ._hostio import HostBuffers
from ..spaces import Box

# reference module-level constants, earl_benchmark/envs/tabletop_manipulation_3obj.py:11-18
initial_states = np.array([[0.0, 0.0, 2.5, 0.0, 2.5, -1.0, 2.5, 1.0, -1., -1.]])
goal_states = np.array([
    [0.0, 0.0, 0.0, -2.0, 0.0, 2.0, -2.5, 1.0, -1., -1.],
])

OBS_DIM, ACT_DIM, MAX_GOALS = 20, 3, 16
_NEVER = 1 << 62


def reset_stream(seed, total_envs, env_offset, num_envs, rows):
    """qpos[0:8] of `rows` successive reset_at_goal resets, float64 [rows, num_envs, 8]: row e, env j of the global batch
    is goal_states[0][:8] + the eight uniforms of env j in draw e of np.random.seed(seed).uniform(-0.3, 0.3,
    8 * total_envs) (tabletop_manipulation_3obj.py:72-76); this shard keeps columns [env_offset, env_offset + num_envs).
    Row e is what the e-th full reset() of a handle without auto_reset draws.  Costs 16 * rows * total_envs draws of the
    legacy Mersenne Twister (made natively) and 64 * rows bytes per env, on the host and on the device."""
    r = rng.NumpyLegacyRandom(int(seed) & 0xFFFFFFFF)
    out = np.empty((rows, num_envs, 8), np.float64)
    for e in range(rows):
        u = r.uniform(-0.3, 0.3, 8 * total_envs).reshape(total_envs, 8)[env_offset:env_offset + num_envs]
        out[e] = goal_states[0][:8] + u
    return out


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


class TabletopManipulation:
    """N independent three-object tabletop envs stepped by one kernel launch.

    Reference-compatible arguments: reward_type, reset_at_goal (tabletop_manipulation_3obj.py:25-27).
    Batched extras: num_envs, device, seed, auto_reset (reset on the device when the horizon fires), reset_stream_rows
    (rows of the pre-drawn reset_at_goal stream of an auto_reset env), eval_stats (per-env episode return and success,
    reduced by eval_stats()), env_offset / total_envs (this shard's slice of a larger job: reset_at_goal draws are made
    for `total_envs` envs and columns [env_offset, env_offset + N) kept), final_obs (with auto_reset: every step's
    info["final_observation"] holds the last observation of each episode the step ended, see step()).
    """

    def __init__(self, reward_type="dense", reset_at_goal=False, num_envs=1, device=None, seed=0, host_io=False,
                 auto_reset=False, reset_stream_rows=64, eval_stats=False, env_offset=0, total_envs=None, final_obs=False):
        if final_obs and not auto_reset:
            raise ValueError("final_obs=True needs auto_reset=True: without it, the observation step() returns on done is the final one")
        if reward_type not in ("sparse", "dense"):
            raise ValueError(f"reward_type must be 'sparse' or 'dense', got {reward_type!r}")
        self._reward_type = reward_type
        self._reset_at_goal = bool(reset_at_goal)
        self.num_envs = int(num_envs)
        self._seed = int(seed)
        self._auto_reset = bool(auto_reset)
        self._reset_stream_rows = int(reset_stream_rows)
        if self._reset_stream_rows < 1:
            raise ValueError("reset_stream_rows must be >= 1")
        self._eval_stats = bool(eval_stats)
        self._keep_final_obs = bool(final_obs)
        self._env_offset = int(env_offset)
        self._total_envs = int(total_envs) if total_envs is not None else self.num_envs + self._env_offset
        if self._env_offset < 0 or self._env_offset + self.num_envs > self._total_envs:
            raise ValueError("envs [env_offset, env_offset + num_envs) must lie inside [0, total_envs)")
        if device is None:
            device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        self.device = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        if self.device.type != "cuda":
            raise ValueError("earl_benchmark_b200 environments live on a CUDA device; there is no CPU path")
        # reference attributes
        self.object_dict = {(0, 0): [2, 3], (0.5, 0.5): [4, 5], (1, 1): [6, 7]}
        self.threshold = 0.4
        self.move_distance = 0.2
        self.initial_state = initial_states.copy()[0]
        self._goal_list = goal_states.copy()
        self.action_space = Box(-1.0, 1.0, (ACT_DIM,), np.float32)
        self.observation_space = Box(-np.inf, np.inf, (OBS_DIM,), np.float32)
        self._goal_table = [g.copy() for g in self._goal_list]
        self._episode_horizon = _NEVER
        self._handle = None
        self._np_random = rng.NumpyLegacyRandom(self._seed & 0xFFFFFFFF)
        self._obs = self._reward = self._done = self._success = self._final_obs = None
        self._host_bufs = None
        self._host_mode = bool(host_io)   # host_io=True: reset() returns numpy like the numpy-driven step()

    def _configure(self, episode_horizon=None, lifelong=None, goal_change_frequency=None):
        if self._handle is not None:
            raise RuntimeError("wrappers must be applied before the env is first reset/stepped")
        if lifelong:
            raise ValueError("LifelongWrapper is not available for the three-object tabletop")
        if episode_horizon is not None:
            self._episode_horizon = int(episode_horizon)

    def _ensure(self):
        if self._handle is not None:
            return
        cfg = _lib.Tt3Config()
        cfg.num_envs, cfg.device = self.num_envs, self.device.index or 0
        cfg.flags = _lib.FLAG_DENSE_REWARD if self._reward_type == "dense" else 0
        cfg.flags |= _lib.FLAG_AUTO_RESET if self._auto_reset else 0
        cfg.flags |= _lib.FLAG_RESET_AT_GOAL if self._reset_at_goal else 0
        cfg.flags |= _lib.FLAG_EVAL_STATS if self._eval_stats else 0
        cfg.flags |= _lib.FLAG_FINAL_OBS if self._keep_final_obs else 0
        cfg.num_goals = MAX_GOALS          # every row is addressable; unused rows repeat row 0 until set
        cfg.episode_horizon = self._episode_horizon
        cfg.threshold, cfg.move_distance, cfg.clip, cfg.success_radius = self.threshold, self.move_distance, 2.8, 0.4
        for k in range(10):
            cfg.initial_state[k] = float(self.initial_state[k])
        if len(self._goal_table) > MAX_GOALS:
            raise ValueError(f"at most {MAX_GOALS} distinct goals")
        for r in range(MAX_GOALS):
            g = self._goal_table[r] if r < len(self._goal_table) else self._goal_table[0]
            for k in range(10):
                cfg.goal_table[r][k] = float(g[k])
        h = C.c_void_p()
        _lib.check(_lib.lib().earl_tt3_create(C.byref(cfg), C.sizeof(cfg), C.byref(h)))
        self._handle = h
        if self._stream_resets():
            rows = reset_stream(self._seed, self._total_envs, self._env_offset, self.num_envs, self._reset_stream_rows)
            _lib.check(_lib.lib().earl_tt3_set_reset_stream(h, rows.ctypes.data, self._reset_stream_rows))
        n, dev = self.num_envs, self.device
        self._obs = torch.empty((n, OBS_DIM), dtype=torch.float32, device=dev)
        self._reward = torch.empty((n,), dtype=torch.float32, device=dev)
        self._done = torch.empty((n,), dtype=torch.uint8, device=dev)
        self._success = torch.empty((n,), dtype=torch.uint8, device=dev)
        self._goal_rows = np.zeros(n, np.int32)
        if self._keep_final_obs:   # rows of envs that have not ended an episode yet hold NaN
            self._final_obs = torch.full((n, OBS_DIM), float("nan"), dtype=torch.float32, device=dev)
            _lib.check(_lib.lib().earl_tt3_set_final_obs(h, self._final_obs.data_ptr()))

    def _stream_resets(self):
        """resets without init_qpos take their qpos from the device's reset stream"""
        return self._auto_reset and self._reset_at_goal

    def close(self):
        if self._handle is not None:
            _lib.lib().earl_tt3_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ goals
    def _mask(self, mask):
        if mask is None:
            return None
        return torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()

    def _rows_for(self, goal):
        g = np.asarray(goal.detach().cpu().numpy() if isinstance(goal, torch.Tensor) else goal, np.float64)
        g = np.broadcast_to(g.reshape(-1, 10) if g.ndim > 1 else g[None, :], (self.num_envs, 10))
        uniq, inv = np.unique(g, axis=0, return_inverse=True)
        rows = np.zeros(len(uniq), np.int32)
        for k, u in enumerate(uniq):
            for r, t in enumerate(self._goal_table):
                if np.array_equal(t, u):
                    rows[k] = r
                    break
            else:
                if self._handle is not None:
                    raise ValueError("custom goals must be registered (reset_goal(goal)) before the env is first used")
                if len(self._goal_table) >= MAX_GOALS:
                    raise ValueError(f"goal table is full ({MAX_GOALS} distinct goals)")
                self._goal_table.append(u.copy())
                rows[k] = len(self._goal_table) - 1
        return rows[inv.reshape(-1)].astype(np.int32)

    def get_next_goal(self):
        """tabletop_manipulation_3obj.py:56-60: np.random.randint(len(goal list)) per env -> [N,10] float64"""
        idx = self._np_random.randint(len(self._goal_list), self.num_envs)
        return self._goal_list[np.asarray(idx, np.int64)]

    def reset_goal(self, goal=None, mask=None):
        if goal is None:
            goal = self.get_next_goal()
        rows = self._rows_for(goal)
        self._ensure()
        m = self._mask(mask)
        sel = np.ones(self.num_envs, bool) if m is None else m.cpu().numpy().astype(bool)
        self._goal_rows[sel] = rows[sel]
        idx = torch.from_numpy(rows).to(self.device)
        _lib.check(_lib.lib().earl_tt3_set_goal(self._handle, _ptr(m), idx.data_ptr(), _stream()))

    @property
    def goal(self):
        """Current goals [N,10] float64 (reference attribute `self.goal`)."""
        self._ensure()
        return np.stack([self._goal_table[r] for r in self._goal_rows])

    # ------------------------------------------------------------------ reset / step
    def reset(self, mask=None, goal_rows=None, init_qpos=None):
        """reset() of every env (or those in `mask`); goal_rows / init_qpos [N,8] override the draws.

        reset_at_goal without init_qpos: a full reset draws np.random.uniform(-0.3, 0.3, 8 * total_envs) and keeps this
        shard's rows; a masked reset draws eight uniforms per selected env, in env order.  On an auto_reset env each
        reset env instead takes its next row of the pre-drawn reset stream (reset_stream())."""
        self._ensure()
        m = self._mask(mask)
        sel = np.ones(self.num_envs, bool) if m is None else m.cpu().numpy().astype(bool)
        # per selected env, in env order: reset_goal() draws np.random.randint(len(goal list)) (one row: consumes
        # nothing), then reset_at_goal adds np.random.uniform(-0.3, 0.3, size=(8,)) to goal[:8]   (:70-73, :82)
        rows = self._goal_rows.copy() if goal_rows is None else np.broadcast_to(np.asarray(goal_rows, np.int32), (self.num_envs,)).copy()
        noisy = init_qpos is None and self._reset_at_goal and not self._stream_resets()
        q = np.zeros((self.num_envs, 8))
        draw = goal_rows is None and len(self._goal_list) > 1
        if goal_rows is None and not draw:
            rows[sel] = 0
        whole = noisy and not draw and m is None    # one draw for the whole job, this shard's slice kept
        if whole:
            lo, n = self._env_offset, self.num_envs
            u = self._np_random.uniform(-0.3, 0.3, 8 * self._total_envs).reshape(self._total_envs, 8)[lo:lo + n]
            q = np.asarray(self._goal_table)[rows, :8] + u
        for i in np.flatnonzero(sel) if (draw or (noisy and not whole)) else ():
            if draw:
                rows[i] = int(self._np_random.randint(len(self._goal_list), 1)[0])
            if noisy:
                q[i] = self._goal_table[rows[i]][:8] + self._np_random.uniform(-0.3, 0.3, 8)
        if noisy:
            init_qpos = q
        iq = None
        if init_qpos is not None:
            iq = torch.as_tensor(np.array(np.broadcast_to(np.asarray(init_qpos, np.float64), (self.num_envs, 8)))).to(self.device)
        self._goal_rows[sel] = rows[sel]
        gi = torch.from_numpy(rows).to(self.device)
        _lib.check(_lib.lib().earl_tt3_reset(self._handle, _ptr(m), gi.data_ptr(), _ptr(iq), 0, _stream()))
        obs = self._get_obs()
        return obs.cpu().numpy() if self._host_mode else obs   # numpy-driven env: numpy out, like its step()

    def step(self, action, out=None):
        """One step of every env.  CUDA float32 [N,3] in -> CUDA tensors out (obs [N,20], reward [N], done [N] bool,
        info; owned by the env, valid until the next step).  numpy / CPU tensor in -> host path, numpy out.
        final_obs=True envs add info["final_observation"] [N,20]: on rows where done is set, the observation the step
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
            _lib.check(_lib.lib().earl_tt3_step(self._handle, a.data_ptr(), obs.data_ptr(), rew.data_ptr(), done.data_ptr(),
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
        _lib.check(_lib.lib().earl_tt3_step_host(self._handle, src.data_ptr(), ho.data_ptr(), hr.data_ptr(), hd.data_ptr(),
                   hs.data_ptr()))
        return HostBuffers.as_numpy(ho, hr, hd, hs, self._final_obs)

    def rollout_into(self, actions, num_steps, obs, reward, done, success=None):
        """`num_steps` back-to-back steps: step t reads actions[t % K], writes slot t % R ([K,N,3]; [R,N,20], [R,N]).
        Not available on final_obs=True envs."""
        if self._keep_final_obs:
            raise RuntimeError("rollout_into does not keep final observations: step() a final_obs=True env")
        self._ensure()
        K, R = actions.shape[0], obs.shape[0]
        assert actions.is_cuda and actions.dtype == torch.float32 and actions.is_contiguous()
        assert obs.shape == (R, self.num_envs, OBS_DIM) and reward.shape == (R, self.num_envs) and done.shape == (R, self.num_envs)
        _lib.check(_lib.lib().earl_tt3_rollout(self._handle, actions.data_ptr(), K, int(num_steps), obs.data_ptr(),
                                               reward.data_ptr(), done.data_ptr(), _ptr(success), R, _stream()))

    # ------------------------------------------------------------------ observation / reward
    def _get_obs(self):
        self._ensure()
        obs = torch.empty((self.num_envs, OBS_DIM), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().earl_tt3_get_obs(self._handle, obs.data_ptr(), _stream()))
        return obs

    def _reward_and_success(self, obs):
        self._ensure()
        host = not (isinstance(obs, torch.Tensor) and obs.is_cuda)
        o = torch.as_tensor(np.asarray(obs, np.float32) if not isinstance(obs, torch.Tensor) else obs)
        o = o.to(self.device, torch.float32).reshape(-1, OBS_DIM).contiguous()
        m = o.shape[0]
        rew = torch.empty((m,), dtype=torch.float32, device=self.device)
        suc = torch.empty((m,), dtype=torch.uint8, device=self.device)
        _lib.check(_lib.lib().earl_tt3_compute_reward(self._handle, o.data_ptr(), m, rew.data_ptr(), suc.data_ptr(), _stream()))
        if host:
            return rew.cpu().numpy(), suc.cpu().numpy().view(np.bool_)
        return rew, suc.view(torch.bool)

    def compute_reward(self, obs):
        return self._reward_and_success(obs)[0]

    def is_successful(self, obs=None):
        if obs is None:
            obs = self._get_obs()
        return self._reward_and_success(obs)[1]

    # ------------------------------------------------------------------ counters / state
    def _counters(self, want_ll=False):
        self._ensure()
        total = C.c_int64()
        interv = torch.empty((self.num_envs,), dtype=torch.int64, device=self.device)
        since = torch.empty((self.num_envs,), dtype=torch.int32, device=self.device)
        _lib.check(_lib.lib().earl_tt3_counters(self._handle, C.byref(total), interv.data_ptr(), since.data_ptr(), _stream()))
        return total.value, interv, since, None

    def eval_stats(self):
        """Device tensor [4] float64: (sum of episode returns, #envs successful at their last step, #envs successful at
        any step of the episode, N), reduced on the device; needs eval_stats=True.  A reset clears an env's statistics.
        Sum it over shards with distributed.all_reduce_eval_stats."""
        self._ensure()
        out = torch.empty((4,), dtype=torch.float64, device=self.device)
        _lib.check(_lib.lib().earl_tt3_eval_stats(self._handle, out.data_ptr(), _stream()))
        return out

    @property
    def launch_count(self):
        return 0 if self._handle is None else int(_lib.lib().earl_tt3_launch_count(self._handle))

    def get_state(self):
        """(qpos [N,8] float64, attached [N] int32: 0 none, 1..3 = object_dict order) as CUDA tensors"""
        self._ensure()
        q = torch.empty((self.num_envs, 8), dtype=torch.float64, device=self.device)
        a = torch.empty((self.num_envs,), dtype=torch.int32, device=self.device)
        _lib.check(_lib.lib().earl_tt3_get_state(self._handle, q.data_ptr(), a.data_ptr(), _stream()))
        return q, a

    def set_state(self, qpos=None, attached=None):
        """reference `set_state(qpos, qvel)` on the eight task coordinates, and / or the attached object"""
        self._ensure()
        q = a = None
        if qpos is not None:
            q = torch.as_tensor(np.array(np.broadcast_to(np.asarray(
                qpos.detach().cpu().numpy() if isinstance(qpos, torch.Tensor) else qpos, np.float64)[..., :8], (self.num_envs, 8)))).to(self.device)
        if attached is not None:
            a = torch.as_tensor(np.broadcast_to(np.asarray(attached, np.int32), (self.num_envs,)).copy()).to(self.device)
        _lib.check(_lib.lib().earl_tt3_set_state(self._handle, _ptr(q), _ptr(a), _stream()))
